#!/usr/bin/env python
"""bench.py — requests/s of the GoFr request hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the CPU restatement of the reference path, host cores
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also store what the last timed step computed

A "step" is one pass of the hot path over one batch of synthetic requests.  Workload at every N: BASELINE config 2 —
16-route GET table, 256-byte JSON struct body, 1 Mi requests per GPU (weak scaling: each rank serves its own
contiguous shard of the request stream; no data-path collective, the sealed route table is broadcast once with NCCL).
  value  : whole-job requests/s with the batch already resident in HBM (CUDA events, max over ranks)
  e2e    : the same through the host-buffer call a user makes (gofr_batch_submit/_wait): pinned host buffers,
           H2D and D2H inside the timed region
  roofline: algorithmic bytes of one launch / its mean CUDA-event duration, against the measured HBM copy peak
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from gofr_b200 import spec as S  # noqa: E402
from gofr_b200 import synth  # noqa: E402

METRIC = "requests_per_sec_256B_json_body"
UNIT = "req/s"
DATE_UNIX = 1789974595
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"


KERNEL_SOURCES = ["gofr_b200/csrc/serve_body.cuh", "gofr_b200/csrc/serve_device.cuh", "gofr_b200/csrc/bind_device.cuh",
                  "gofr_b200/csrc/serve_slots_kernel.cu", "gofr_b200/csrc/serve_slots_wide_kernel.cu", "gofr_b200/csrc/serve_values_kernel.cu", "gofr_b200/csrc/serve_slots_values_kernel.cu", "gofr_b200/csrc/value_device.cuh", "gofr_b200/csrc/float_device.cuh", "gofr_b200/csrc/serve_kernel.cu", "gofr_b200/csrc/tile_common.cuh",
                  "gofr_b200/csrc/table_format.h"]


def kernel_source_hash():
    """SHA-256 over what decides the serve kernels' binaries: their sources and headers, the compiler flags and the list of
    translation units built with the 256-bit sector store (not the whole build script: adding an unrelated kernel to the
    build must not invalidate a capture of this one)."""
    import hashlib
    from gofr_b200 import _build
    h = hashlib.sha256()
    for f in KERNEL_SOURCES:
        with open(os.path.join(ROOT, f), "rb") as fh:
            h.update(fh.read())
    h.update(repr((_build.NVCC_FLAGS, sorted(x for x in _build.SECTOR256 if x.startswith("serve")))).encode())
    return h.hexdigest()


def profiled_traffic(layout="slots"):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the headline kernel on this exact workload, from an
    `ncu --set full` capture — reported only when the capture was taken from the kernel sources that are being run now
    (profiles/r02/traffic.json records their SHA-256; a stale capture yields null, never an old number)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02", "traffic.json")) as f:
            t = json.load(f)
        ent = t.get(layout)
        if not ent or ent.get("source_sha256") != kernel_source_hash():
            return None
        return float(ent["dram_bytes_read"]) + float(ent["dram_bytes_write"])
    except Exception:
        return None


class ClockSampler:
    """Samples SM clocks and throttle reasons DURING the timed region.  NVML in-process (one query takes tens of
    microseconds, so even a few-millisecond region gets many samples); `nvidia-smi -lms` as a fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index
        self.nvml = None
        self.stop_flag = False
        self.samples = []  # (sm_mhz, reasons bitmask)
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes CUDA_VISIBLE_DEVICES; map through the UUID torch reports when possible
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
                for cand in ("GPU-" + uuid, uuid):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        h = None
            except Exception:
                h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nvml, self.h = pynvml, h
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _poll(self):
        nv, h = self.nvml, self.h
        while not self.stop_flag:
            try:
                self.samples.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                     int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))))
            except Exception:
                break
            time.sleep(0.0005)

    def start(self):
        if self.nvml is not None:
            self.stop_flag = False
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.t.join(timeout=1.0)
            nv = self.nvml
            bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                    "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                    "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                    "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
            sm = [s[0] for s in self.samples]
            seen = 0
            for s in self.samples:
                seen |= s[1]
            reasons = sorted(k for k, b in bits.items() if seen & b)
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


DUMP_ROWS = 16384  # responses --dump-outputs stores byte for byte: 16 Ki 528-byte slots as float32 are 35 MB


def dump_outputs(path, n, width, slots, resp):
    """--dump-outputs: what the resident path handed its caller in the last timed step (`slots` = (out, out_len, meta) of
    the slot layout, else the packed `resp`), for comparing two builds output for output.  A fixed, seeded sample of
    DUMP_ROWS requests (all of them when there are fewer): their response bytes (zero past each response's end), lengths
    and meta words, in the same form for both layouts.  float32 holds every byte and length exactly, float64 every uint32
    meta word and request index."""
    import torch
    k = min(n, DUMP_ROWS)
    idx = np.sort(np.random.default_rng(synth.SEED).choice(n, k, replace=False))
    i = torch.from_numpy(idx).to(resp.out.device)
    if slots is not None:
        s_out, s_len, s_meta = slots
        buf, start, length, meta = s_out, i * width, s_len[i].long(), s_meta[i]
    else:
        off = resp.out_off.long() & 0xFFFFFFFF
        buf, start, length, meta = resp.out, off[i], off[i + 1] - off[i], resp.meta[i]
    assert bool((length <= width).all()), "a response longer than the dump's row width"
    col = torch.arange(width, device=buf.device)
    keep = col < length[:, None]
    rows = torch.where(keep, buf[torch.where(keep, start[:, None] + col, 0)], 0)
    arrays = {"request_index": idx.astype(np.float64), "response_bytes": rows.cpu().numpy().astype(np.float32),
              "response_len": length.cpu().numpy().astype(np.float32),
              "meta": (meta.long() & 0xFFFFFFFF).cpu().numpy().astype(np.float64)}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def bind_to_gpu_numa(device: int):
    import ctypes as C
    from gofr_b200 import _abi
    node = C.c_int(-1)
    rc = _abi.lib().gofr_bind_host_thread(device, C.byref(node))
    d = {"bound": rc == 0, "node": node.value if node.value >= 0 else None, "cpus": len(os.sched_getaffinity(0))}
    if rc != 0:
        d["why"] = _abi.lib().gofr_last_error().decode(errors="replace")
    return d


def link_floor_ms(device, h2d_bytes: int, d2h_bytes: int, steps: int = 5):
    """The platform floor of one end-to-end step: the step's H2D and D2H bytes moved concurrently between pinned host
    buffers and HBM, no kernel (CUDA events on two streams; the caller takes the max over ranks)."""
    import torch
    h_in = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    d_in = torch.empty(h2d_bytes, dtype=torch.uint8, device=device)
    d_out = torch.zeros(d2h_bytes, dtype=torch.uint8, device=device)
    s1, s2 = torch.cuda.Stream(device), torch.cuda.Stream(device)

    def step():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)
        s1.synchronize(); s2.synchronize()
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / steps * 1e3


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def cpu_quota():
    """CPUs' worth of time the cgroup grants this container per period (cgroup v2 cpu.max / v1 cfs_quota_us), or None.
    The GPU boxes of this pool show 128 logical CPUs and a quota of 16: more runnable threads than the quota only get
    the whole container throttled for the rest of each 100 ms period."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def pick_cpu_threads(run_with):
    """The thread count the CPU arm gets: whichever of {all logical CPUs, the cgroup quota} serves one pass faster."""
    import math
    ncpu = os.cpu_count() or 1
    cands = [ncpu]
    q = cpu_quota()
    if q and math.ceil(q) < ncpu:
        cands.append(max(1, math.ceil(q)))
    best, best_rate = cands[0], None
    for c in cands:
        run_with(c)                       # touch the pages / spin the threads up
        # at least half a second per candidate: a single pass can fit into what is left of one 100 ms quota period and
        # look unthrottled
        t0 = time.perf_counter()
        passes = 0
        while passes < 3 or time.perf_counter() - t0 < 0.5:
            run_with(c)
            passes += 1
        rate = passes / (time.perf_counter() - t0)
        if best_rate is None or rate > best_rate:
            best, best_rate = c, rate
    return best, q


def run_reference(args):
    """The reference arm: the CPU restatement of the reference's Go path (oracle/, kind "port" — no Go toolchain
    exists in this image, so the reference itself cannot be built) on all host cores, same workload and metric."""
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    from tests import oracle as O
    n = args.ref_requests
    spec = synth.config2_spec(S.FRAME_WIRE)
    batch = synth.config2_batch(n)
    table = O.OracleTable(spec)
    date = S.http_date(DATE_UNIX)
    cap = n * 640 + 4096
    out = np.zeros(cap, dtype=np.uint8)
    off = np.zeros(n + 1, dtype=np.uint32)
    meta = np.zeros(n, dtype=np.uint32)

    def step(threads=None):
        rc = O.lib().orc_serve(table._t, batch.desc.ctypes.data, batch.trace_ids.ctypes.data, batch.arena.ctypes.data,
                               n, date, out.ctypes.data, cap, off.ctypes.data, meta.ctypes.data, threads or cores)
        assert rc == 0

    cores, quota = pick_cpu_threads(step)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    sample = (f"{n} requests per step of the config-2 stream, {cores} pthreads of {os.cpu_count()} logical CPUs"
              f" (cgroup CPU quota: {quota if quota else 'none'}), in-memory (no sockets, no logging)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(n, args.gpus, args),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "cpu_quota": quota},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def workload_config(n, gpus, args):
    """The `config` object of both arms (this repo's and `--impl reference`): identical by construction."""
    return {"workload": "BASELINE config 2: 16-route GET table, 256B JSON struct body (521B full HTTP/1.1 response, wire "
                        "framing), %d requests per step per worker (GPU rank / CPU arm)" % n,
            "requests_per_step_per_worker": n, "frame_mode": "wire", "routes": 16,
            "parallelism": f"dp{gpus} (requests sharded, no data-path collective)",
            "l2": "inputs+outputs per step (~%.2f GB) %s the 126 MB L2" % (n * 793 / 1e9, "exceed" if n * 793 > 126e6 else "DO NOT exceed"),
            "resident_layout": ("slots: response i in its own 528-byte slot (gofr_serve_device_slots)" if args.layout == "slots" else "packed offsets (gofr_serve_device)"),
            "e2e_layout": ("slots (gofr_batch_submit_slots)" if args.e2e_layout == "slots" else "packed offsets (gofr_batch_submit)")}


def run_secondary(args):
    """Resident-only measurements of the other BASELINE configs (1 GPU): kernel time per launch and requests/s."""
    import torch
    from gofr_b200 import _abi
    from gofr_b200.engine import Engine
    from gofr_b200.table import Table
    from tests import oracle as O
    date = S.http_date(DATE_UNIX)
    w = args.workload
    n = {"config3": 65536, "config4": 262144, "config5": 1 << 20, "proto": 1 << 20, "reqlog": 1 << 18, "http": 1 << 20}[w] if args.requests == (1 << 20) and w not in ("config5", "proto") else args.requests
    cpu = None
    cpu_fn = cpu_what = e2e_step = None
    xfer_in, xfer_out, e2e_bytes = [], [], None
    if w == "reqlog":
        # the RequestLog line of middleware.Logging for the config-2 stream (SURVEY.md §8f rank 1)
        lb = synth.reqlog_batch(n)
        eng = Engine(Table(synth.config1_spec()), 0)
        eng.set_timing(True)
        d_desc = torch.from_numpy(lb.desc.view(np.uint8).reshape(-1).copy()).cuda()
        d_ids = torch.from_numpy(lb.trace_ids.reshape(-1).copy()).cuda()
        d_arena = torch.from_numpy(np.concatenate([lb.arena, np.zeros(48, np.uint8)])).cuda()
        cap = 400 * n + 6 * int(lb.arena.size)
        d_out = torch.zeros(cap + 64, dtype=torch.uint8, device="cuda")
        d_ooff = torch.zeros(n + 1, dtype=torch.int32, device="cuda")

        def step():
            eng.request_log_resident(d_desc, d_ids, d_arena, n, d_out, cap, d_ooff)
        in_bytes = lb.input_bytes() - 8 * n  # the generic "+ 8 * n" below counts offsets + meta; here only 4-byte offsets leave
        in_bytes += 4 * n
        get_out = lambda: int(d_ooff[n].item())
        cpu_fn, cpu_what = (lambda: (O.request_log(lb), n)[1]), "scalar C restatement (oracle/orc_reqlog.c), 1 thread"
        xfer_in, xfer_out = [d_desc, d_ids, d_arena], [(d_out, lambda: int(d_ooff[n].item())), (d_ooff, None)]
    elif w == "http":
        # raw HTTP/1.1 request messages of the config-2 stream → descriptors + arena (SURVEY.md §8f rank 2)
        n = args.requests if args.requests != (1 << 20) else (1 << 20)
        raw, off = synth.http_messages(n)
        eng = Engine(Table(synth.config1_spec()), 0)
        eng.set_timing(True)
        d_raw = torch.from_numpy(np.concatenate([raw, np.zeros(32, np.uint8)])).cuda()
        d_off = torch.from_numpy(off.view(np.int32)).cuda()
        d_desc = torch.zeros(n * 16, dtype=torch.uint8, device="cuda")
        d_arena = torch.zeros(int(raw.size) + 48, dtype=torch.uint8, device="cuda")
        d_status = torch.zeros(n, dtype=torch.int32, device="cuda")
        d_spans = torch.zeros((n, 6), dtype=torch.int64, device="cuda")
        st = torch.cuda.current_stream().cuda_stream

        def step():
            _abi.check(_abi.lib().gofr_http_parse_device(eng._e, d_raw.data_ptr(), d_off.data_ptr(), n, d_desc.data_ptr(),
                                                         d_arena.data_ptr(), d_status.data_ptr(), d_spans.data_ptr(), st), "http")
        step()
        torch.cuda.synchronize()
        dd = d_desc.cpu().numpy().view(S.DESC_DTYPE)
        assert int((d_status != 0).sum().item()) == 0
        written = int(((dd["path_len"].astype(np.int64) + dd["query_len"] + 3) & ~3).sum() + dd["data_len"].astype(np.int64).sum())
        in_bytes = int(raw.size) + 4 * (n + 1) + 16 * n + 4 * n + 48 * n - 8 * n  # the generic "+ 8 * n" is added below
        get_out = lambda: written
        cpu_fn, cpu_what = (lambda: (O.http_parse(raw, off), n)[1]), "scalar C restatement (oracle/orc_http.c), 1 thread"
        xfer_in, xfer_out = [d_raw, d_off], [(d_desc, None), (d_arena, lambda: int(raw.size)), (d_status, None)]
    elif w == "proto":
        # rows of a 9-field message (string, int64, sint32, bool, double, bytes, fixed32, int32, string) → gRPC frames
        rng = np.random.default_rng(synth.SEED)
        fields = [S.ProtoField(1, S.PB_STRING), S.ProtoField(2, S.PB_INT64), S.ProtoField(3, S.PB_SINT32), S.ProtoField(4, S.PB_BOOL),
                  S.ProtoField(5, S.PB_DOUBLE), S.ProtoField(7, S.PB_BYTES), S.ProtoField(9, S.PB_FIXED32), S.ProtoField(300, S.PB_INT32),
                  S.ProtoField(301, S.PB_STRING)]
        # rows built vectorised: 12 fixed words + a 16-byte name + 8 bytes + a 12-byte tag = 84 bytes each
        fixed = np.zeros((n, 12), dtype=np.uint32)
        r = rng.integers(0, 1 << 62, (n, 4), dtype=np.int64)
        fixed[:, 0] = 16
        fixed[:, 1] = (r[:, 0] & 0xFFFFFFFF).astype(np.uint32); fixed[:, 2] = ((r[:, 0] >> 32) & 0x3FFFFF).astype(np.uint32)
        fixed[:, 3] = (r[:, 1] % 2001 - 1000).astype(np.int32).view(np.uint32)
        fixed[:, 4] = (r[:, 1] >> 20 & 1).astype(np.uint32)
        dbl = ((r[:, 2] % 100000) / 8.0).astype(np.float64).view(np.uint64)
        fixed[:, 5] = (dbl & 0xFFFFFFFF).astype(np.uint32); fixed[:, 6] = (dbl >> 32).astype(np.uint32)
        fixed[:, 7] = 8
        fixed[:, 8] = (r[:, 3] & 0xFFFFFFFF).astype(np.uint32)
        fixed[:, 9] = (-(r[:, 3] >> 40) % 50000).astype(np.int32).view(np.uint32)
        fixed[:, 10] = 12
        tail = (rng.integers(0, 26, (n, 36), dtype=np.uint8) + 97).astype(np.uint8)
        rows = np.concatenate([fixed.view(np.uint8).reshape(n, 48), tail], axis=1).reshape(-1)
        rows = np.concatenate([rows, np.zeros(64, np.uint8)])
        off = (np.arange(n + 1, dtype=np.uint64) * 84).astype(np.uint32)
        eng = Engine(Table(synth.config1_spec()), 0)
        eng.set_timing(True)
        # parity of the bench's own input (first 4096 rows)
        o_out, o_off, o_meta = O.proto_encode(fields, rows, off[:4097])
        d_in = torch.from_numpy(rows).cuda()
        d_off = torch.from_numpy(off.view(np.int32)).cuda()
        cap = n * 128
        d_out = torch.zeros(cap + 64, dtype=torch.uint8, device="cuda")
        d_ooff = torch.zeros(n + 1, dtype=torch.int32, device="cuda")
        d_meta = torch.zeros(n, dtype=torch.int32, device="cuda")
        st = torch.cuda.current_stream().cuda_stream
        ft = (_abi.ProtoField * len(fields))(*[_abi.ProtoField(f.number, f.type) for f in fields])

        def step():
            _abi.check(_abi.lib().gofr_proto_encode_device(eng._e, ft, len(fields), d_in.data_ptr(), d_off.data_ptr(), n,
                                                           d_out.data_ptr(), cap, d_ooff.data_ptr(), d_meta.data_ptr(), st), "proto")
        step()
        torch.cuda.synchronize()
        assert d_out[:int(o_off[4096])].cpu().numpy().tobytes() == o_out[:int(o_off[4096])].tobytes(), "bench output differs from the oracle"
        in_bytes = int(off[n]) + 4 * (n + 1)
        get_out = lambda: int(d_ooff[n].item())
        m_cpu = min(n, 1 << 18)
        cpu_fn, cpu_what = (lambda: (O.proto_encode(fields, rows, off[:m_cpu + 1]), m_cpu)[1]), "scalar C restatement (oracle/orc_proto.c), 1 thread"
        xfer_in, xfer_out = [d_in, d_off], [(d_out, lambda: int(d_ooff[n].item())), (d_ooff, None), (d_meta, None)]
    elif w == "config5":
        frames, off = synth.config5_frames(n)
        eng = Engine(Table(synth.config1_spec()), 0)
        eng.set_timing(True)
        d_in = torch.from_numpy(np.concatenate([frames, np.zeros(64, np.uint8)])).cuda()
        d_off = torch.from_numpy(off.view(np.int32)).cuda()
        cap = int(frames.size) + 40 * n
        d_out = torch.zeros(cap + 64, dtype=torch.uint8, device="cuda")
        d_ooff = torch.zeros(n + 1, dtype=torch.int32, device="cuda")
        d_meta = torch.zeros(n, dtype=torch.int32, device="cuda")
        st = torch.cuda.current_stream().cuda_stream

        def step():
            _abi.check(_abi.lib().gofr_grpc_hello_device(eng._e, d_in.data_ptr(), d_off.data_ptr(), n, d_out.data_ptr(), cap,
                                                         d_ooff.data_ptr(), d_meta.data_ptr(), st), "grpc")
        in_bytes = int(off[n]) + 4 * (n + 1)
        get_out = lambda: int(d_ooff[n].item())
        cpu_threads = max(1, int(cpu_quota() or os.cpu_count() or 1))
        cpu_fn, cpu_what = (lambda: (O.grpc_hello(frames, off, cpu_threads), n)[1]), f"C restatement (oracle/orc_grpc.c), {cpu_threads} pthreads"
        xfer_in, xfer_out = [d_in, d_off], [(d_out, lambda: int(d_ooff[n].item())), (d_ooff, None), (d_meta, None)]
    else:
        spec, batch = {"config3": (synth.config3_spec(), lambda: synth.config3_batch(n)),
                       "config4": (synth.config4_spec(), lambda: synth.config4_batch(n))}[w]
        batch = batch()
        eng = Engine(Table(spec), 0)
        eng.set_timing(True)
        db = eng.upload(batch)
        o1, f1, _ = O.OracleTable(spec).serve(batch, date)
        resp = eng.alloc_responses(n, int(f1[n]) + 4096)

        if args.layout == "slots":
            slot = 1024
            s_out = torch.empty(n * slot, dtype=torch.uint8, device="cuda")
            s_len = torch.zeros(n, dtype=torch.int32, device="cuda")
            s_meta = torch.zeros(n, dtype=torch.int32, device="cuda")

            def step():
                eng.serve_device_slots(db, date, slot, out=s_out, out_len=s_len, meta=s_meta)
            get_out = lambda: int(s_len.sum().item())
        else:
            def step():
                eng.serve_device(db, date, resp)
            get_out = lambda: int(resp.out_off[n].item())
        in_bytes = batch.input_bytes()
        ot = O.OracleTable(spec)
        cpu_threads = max(1, int(cpu_quota() or os.cpu_count() or 1))
        m_cpu = min(n, 1 << 18)
        sbatch = batch.slice(0, m_cpu)
        cpu_fn, cpu_what = (lambda: (ot.serve(sbatch, date, nthreads=cpu_threads), m_cpu)[1]), f"C restatement (oracle/gofr_oracle.c), {cpu_threads} pthreads"
        from gofr_b200.engine import pin_batch, pinned_array
        hb = pin_batch(batch)
        eslot = 1024
        h_out, h_len, h_meta = pinned_array(n * eslot), pinned_array(4 * n, np.uint32), pinned_array(4 * n, np.uint32)
        e2e_step = lambda: eng.serve_host_slots(hb, date, eslot, h_out, h_len, h_meta)
        e2e_bytes = (n * 32 + int(batch.arena_span()), n * eslot + 8 * n)
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    eng.kernel_time_ms(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / args.steps
    kms, kl = eng.kernel_time_ms(reset=True)
    out_bytes = get_out()
    algo = in_bytes + out_bytes + 8 * n
    peak, src = hbm_peak()
    # ---- end to end: pinned host buffers -> HBM -> kernel -> pinned host buffers, every step ----
    if e2e_step is None:
        h_in = [t.cpu().pin_memory() for t in xfer_in]
        outs = [(d, (f() if f else d.numel() * d.element_size())) for d, f in xfer_out]
        h_outs = [torch.empty(nb, dtype=torch.uint8).pin_memory() for _, nb in outs]

        def e2e_step():
            for h, d in zip(h_in, xfer_in):
                d.copy_(h, non_blocking=True)
            step()
            for (d, nb), h in zip(outs, h_outs):
                h.copy_(d.view(torch.uint8).reshape(-1)[:nb], non_blocking=True)
            torch.cuda.synchronize()
        e2e_bytes = (sum(t.numel() * t.element_size() for t in xfer_in), sum(nb for _, nb in outs))
    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_dt = (time.perf_counter() - t0) / args.steps
    e2e = {"value": n / e2e_dt, "unit": UNIT, "ms_per_step": e2e_dt * 1e3, "h2d_bytes_per_step": int(e2e_bytes[0]), "d2h_bytes_per_step": int(e2e_bytes[1])}
    # ---- CPU restatement beside it: bounded sample, at least ~1 s ----
    if cpu_fn is not None:
        cpu_fn()
        t0 = time.perf_counter()
        units = 0
        while time.perf_counter() - t0 < 1.0:
            units += cpu_fn()
        cpu = {"value": units / (time.perf_counter() - t0), "unit": UNIT, "kind": "port", "sample": f"passes over (a prefix of) the same input for >= 1 s: {cpu_what}"}
    print(json.dumps({"metric": "requests_per_sec", "workload": w, "e2e": e2e, "layout": args.layout if w in ("config3", "config4") else None, "value": n / (ms / 1e3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": ms, "requests": n, "out_bytes": out_bytes, "data": "synthetic",
                      "roofline": {"bound": "hbm", "achieved": algo / (kms / kl / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                                   "frac": algo / (kms / kl / 1e3) / 1e9 / peak, "algorithmic_bytes_per_request": algo / n,
                                   "kernel_ms_per_launch": kms / kl},
                      **({"cpu_baseline": cpu} if cpu else {})}))
    return 0


def sharded_config4(eng_factory, rank, world, dev, barrier, reduce_max, steps, per_gpu=1 << 18):
    """BASELINE config 4 ("mixed 64-route GET/POST with the 3-deep middleware chain, 4xB200 shard"): the 64-route table is
    sealed on rank 0 and broadcast (NCCL), every rank serves its contiguous shard of ONE request stream, resident and
    through host buffers; parity of a sample of the rank's shard against the oracle run on exactly those requests."""
    import torch
    from gofr_b200.engine import pin_batch, pinned_array
    from tests import oracle as O
    date = S.http_date(DATE_UNIX)
    spec = synth.config4_spec()
    eng = eng_factory(spec)
    eng.set_timing(True)
    n = per_gpu
    batch = synth.config4_batch(n, start=rank * n)
    db = eng.upload(batch)
    slot = 1024
    s_out = torch.zeros(n * slot, dtype=torch.uint8, device=dev)
    s_len = torch.zeros(n, dtype=torch.int32, device=dev)
    s_meta = torch.zeros(n, dtype=torch.int32, device=dev)
    step = lambda: eng.serve_device_slots(db, date, slot, out=s_out, out_len=s_len, meta=s_meta)
    for _ in range(3):
        step()
    barrier()
    eng.kernel_time_ms(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = reduce_max(e0.elapsed_time(e1)) / steps
    kms, kl = eng.kernel_time_ms(reset=True)
    # parity: the first 4096 requests of this rank's shard against the oracle on the same requests
    m = 4096
    o1, f1, m1 = O.OracleTable(spec).serve(batch.slice(0, m), date)
    ln = s_len[:m].cpu().numpy().view(np.uint32)
    # (recorded, not asserted: an assertion on one rank would leave the others waiting at the next barrier)
    bad = 0 if (np.array_equal(ln, np.diff(f1.astype(np.int64)).astype(np.uint32)) and
                np.array_equal(s_meta[:m].cpu().numpy().view(np.uint32), m1)) else 1
    so = s_out[:m * slot].cpu().numpy().reshape(m, slot)
    if not bad:
        for i in range(m):
            L = int(ln[i])
            if L <= slot and so[i, :L].tobytes() != o1[int(f1[i]):int(f1[i]) + L].tobytes():
                bad = 1
                break
    out_bytes = int(s_len.sum().item())
    # end to end through host buffers
    hb = pin_batch(batch)
    h_out, h_len, h_meta = pinned_array(n * slot), pinned_array(4 * n, np.uint32), pinned_array(4 * n, np.uint32)
    for _ in range(2):
        eng.serve_host_slots(hb, date, slot, h_out, h_len, h_meta)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        eng.serve_host_slots(hb, date, slot, h_out, h_len, h_meta)
    barrier()
    dt = reduce_max(time.perf_counter() - t0) / steps
    if not np.array_equal(h_len[:m], ln):
        bad = 1
    bad = int(reduce_max(float(bad)))
    algo = batch.input_bytes() + out_bytes + 8 * n
    peak, _ = hbm_peak()
    eng.close()
    return {"workload": "BASELINE config 4: 64 mixed routes (GET/POST, OPTIONS / 404 / 301 / HEAD traffic), %d requests per GPU, table broadcast from rank 0" % n,
            "value": n * world / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "kernel_ms_per_launch": kms / max(kl, 1),
            "roofline_frac": algo / (kms / max(kl, 1) / 1e3) / 1e9 / peak, "algorithmic_bytes_per_request": algo / n,
            "e2e": {"value": n * world / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "h2d_bytes_per_step": n * 32 + int(batch.arena_span()), "d2h_bytes_per_step": n * slot + 8 * n},
            "parity": (f"first {m} responses of every rank's shard byte-identical to the oracle run on those requests" if not bad else
                       "FAILED: some rank's shard differs from the oracle")}


def sharded_config5(eng, rank, world, dev, barrier, reduce_max, steps, per_gpu=1 << 20):
    """BASELINE config 5 ("gRPC unary protobuf encode path, 1M req, 8xB200 with NCCL route-table broadcast"): every rank
    decodes / answers / encodes its contiguous shard of one HelloRequest frame stream (the engine's table came from the
    NCCL broadcast at start-up); parity of a sample against the oracle."""
    import torch
    from gofr_b200 import _abi
    from tests import oracle as O
    n = per_gpu
    frames, off = synth.config5_frames(n, start=rank * n)
    d_in = torch.from_numpy(np.concatenate([frames, np.zeros(64, np.uint8)])).to(dev)
    d_off = torch.from_numpy(off.view(np.int32)).to(dev)
    cap = int(frames.size) + 40 * n
    d_out = torch.zeros(cap + 64, dtype=torch.uint8, device=dev)
    d_ooff = torch.zeros(n + 1, dtype=torch.int32, device=dev)
    d_meta = torch.zeros(n, dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    step = lambda: _abi.check(_abi.lib().gofr_grpc_hello_device(eng._e, d_in.data_ptr(), d_off.data_ptr(), n, d_out.data_ptr(), cap,
                                                                  d_ooff.data_ptr(), d_meta.data_ptr(), st), "grpc")
    for _ in range(3):
        step()
    barrier()
    eng.kernel_time_ms(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = reduce_max(e0.elapsed_time(e1)) / steps
    kms, kl = eng.kernel_time_ms(reset=True)
    m = 8192
    o_out, o_off, o_meta = O.grpc_hello(frames, off[:m + 1])
    g_off = d_ooff[:m + 1].cpu().numpy().view(np.uint32)
    bad = 0 if (np.array_equal(g_off, o_off) and d_out[:int(o_off[m])].cpu().numpy().tobytes() == o_out[:int(o_off[m])].tobytes()) else 1
    bad = int(reduce_max(float(bad)))
    out_bytes = int(d_ooff[n].item())
    algo = int(off[n]) + 4 * (n + 1) + out_bytes + 8 * n
    peak, _ = hbm_peak()
    return {"workload": "BASELINE config 5: gRPC unary SayHello, %d length-prefixed HelloRequest frames per GPU" % n,
            "value": n * world / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "kernel_ms_per_launch": kms / max(kl, 1),
            "roofline_frac": algo / (kms / max(kl, 1) / 1e3) / 1e9 / peak, "algorithmic_bytes_per_request": algo / n,
            "parity": (f"first {m} response frames of every rank's shard byte-identical to the oracle" if not bad else
                       "FAILED: some rank's shard differs from the oracle")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--requests", type=int, default=1 << 20, help="requests per GPU per step")
    ap.add_argument("--ref-requests", type=int, default=1 << 20, help="requests per step of the CPU reference arm")
    ap.add_argument("--cpu-sample", type=int, default=1 << 19, help="requests in the cpu_baseline sample")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer measurement (default: --steps)")
    ap.add_argument("--chunk", type=int, default=65536)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="leave the rank's threads and pinned buffers wherever the OS puts them")
    ap.add_argument("--no-extras", action="store_true", help="skip the sharded config-4 (4 GPUs) / config-5 (8 GPUs) legs")
    ap.add_argument("--extras-timeout", type=int, default=240, help="seconds the sharded legs may take before the headline line is printed without them")
    ap.add_argument("--e2e-layout", default="slots", choices=["packed", "slots"],
                    help="end-to-end measurement: gofr_batch_submit (packed offsets, device-driven egress) or "
                         "gofr_batch_submit_slots (one slot per response, plain async copies)")
    ap.add_argument("--layout", default="slots", choices=["packed", "slots"],
                    help="resident measurement: packed offsets (gofr_serve_device) or one 528-byte slot per response "
                         "(gofr_serve_device_slots)")
    ap.add_argument("--workload", default="config2", choices=["config2", "config3", "config4", "config5", "proto", "reqlog", "http"],
                    help="config2 is the BASELINE metric line; the others are secondary measurements (resident only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's shard; a seeded sample of "
                         "%d responses, their lengths and meta words) as DIR/<name>.npy in float32 / float64" % DUMP_ROWS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.workload != "config2"):
        ap.error("--dump-outputs stores the outputs of the config-2 headline path only")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from gofr_b200.engine import Engine, pin_batch, pinned_array
    from gofr_b200.table import Table

    rank, world, local = dist_env()
    if args.workload != "config2":
        return run_secondary(args)
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: gofr_b200 has no CPU path"}))
        return 2
    # Before anything is pinned: this rank's threads and the pages they touch go to the NUMA node its GPU hangs off
    # (GPU0-3 and GPU4-7 sit on different sockets on the 8-GPU boxes; unbound, every rank's pinned buffers can land on
    # one socket and half of the PCIe traffic crosses the inter-socket link).
    cpus_before_bind = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local) if not args.no_numa_bind else {"bound": False, "node": None, "why": "--no-numa-bind"}
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- route table: sealed on rank 0, broadcast as bytes over NCCL, deserialised everywhere ----
    from gofr_b200 import dist as gd
    image = Table(synth.config2_spec(S.FRAME_WIRE)).serialize() if rank == 0 else None
    image = gd.broadcast_table_image(image, rank, dev)
    table = Table(image=image)
    eng = Engine(table, local)
    eng.set_chunk(args.chunk)
    eng.set_timing(True)  # CUDA events around every kernel launch of this engine (roofline.achieved)

    n = args.requests
    date = S.http_date(DATE_UNIX)
    batch = synth.config2_batch(n, start=rank * n)  # this rank's shard of the stream
    out_bytes = n * synth.C2_WIRE_BYTES
    db = eng.upload(batch)
    resp = eng.alloc_responses(n, out_bytes + 4096)
    # algorithmic bytes of one launch: every input byte read once, every output byte written once
    algo_bytes = batch.input_bytes() + out_bytes + 4 * (n + 1) + 4 * n

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- resident measurement (`value`, roofline) ----
    slot = (synth.C2_WIRE_BYTES + 15) & ~15
    if args.layout == "slots":
        s_out = torch.empty(n * slot, dtype=torch.uint8, device=dev)
        s_len = torch.zeros(n, dtype=torch.int32, device=dev)
        s_meta = torch.zeros(n, dtype=torch.int32, device=dev)

        def serve_resident():
            eng.serve_device_slots(db, date, slot, out=s_out, out_len=s_len, meta=s_meta)
    else:
        def serve_resident():
            eng.serve_device(db, date, resp)
    for _ in range(args.warmup):
        serve_resident()
    barrier()
    assert not eng.overflowed()
    eng.kernel_time_ms(reset=True)
    launches0 = eng.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        serve_resident()
    ev1.record()
    barrier()
    ms = reduce_max(ev0.elapsed_time(ev1))
    clocks = sampler.stop()
    kernel_ms, kernel_launches = eng.kernel_time_ms(reset=True)
    launches = eng.launch_count() - launches0
    value = n * world * args.steps / (ms / 1e3)
    per_launch_ms = kernel_ms / max(kernel_launches, 1)
    achieved = algo_bytes / (per_launch_ms / 1e3) / 1e9
    peak, peak_src = hbm_peak()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, n, slot, (s_out, s_len, s_meta) if args.layout == "slots" else None, resp)

    # the other layout, measured the same way (reported beside the headline number, not instead of it)
    alt = None
    if args.layout == "slots":
        for _ in range(args.warmup):
            eng.serve_device(db, date, resp)
        barrier()
        eng.kernel_time_ms(reset=True)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(args.steps):
            eng.serve_device(db, date, resp)
        a1.record()
        barrier()
        alt_ms = reduce_max(a0.elapsed_time(a1))
        akm, akl = eng.kernel_time_ms(reset=True)
        alt = {"layout": "packed (gofr_serve_device: offsets chained across tiles by the look-back)",
               "value": n * world * args.steps / (alt_ms / 1e3), "kernel_ms_per_launch": akm / max(akl, 1),
               "frac": algo_bytes / (akm / max(akl, 1) / 1e3) / 1e9 / peak}
    # spot check inside the bench: sizes are what the workload says
    if args.layout == "slots":
        assert bool((s_len == synth.C2_WIRE_BYTES).all()), "unexpected response size"
        k = 4096
        a = s_out[:k * slot].view(k, slot)[:, :synth.C2_WIRE_BYTES].reshape(-1)
        assert bool((a == resp.out[:k * synth.C2_WIRE_BYTES]).all()), "slot layout and packed layout disagree"
    else:
        pass
    off = resp.out_off.cpu().numpy().view(np.uint32)
    assert int(off[n]) == out_bytes, "unexpected response size"

    # ---- end-to-end measurement: host buffers through gofr_batch_submit/_wait ----
    e2e = None
    if not args.no_e2e:
        hb = pin_batch(batch)
        ksteps = args.e2e_steps or args.steps
        h2d = n * 32 + int(batch.arena_span())
        if args.e2e_layout == "slots":
            h_out = pinned_array(n * slot)
            h_len = pinned_array(4 * n, np.uint32)
            h_meta = pinned_array(4 * n, np.uint32)
            for _ in range(args.warmup):
                eng.serve_host_slots(hb, date, slot, h_out, h_len, h_meta)
            assert bool((h_len == synth.C2_WIRE_BYTES).all())
            barrier()
            t0 = time.perf_counter()
            for _ in range(ksteps):
                eng.serve_host_slots(hb, date, slot, h_out, h_len, h_meta)
            barrier()
            dt = reduce_max(time.perf_counter() - t0)
            d2h = n * slot + 4 * n + 4 * n
            # the last host result must match the resident (packed) one byte for byte, response by response
            k = 8192
            dev_out = resp.out[:k * synth.C2_WIRE_BYTES].cpu().numpy().reshape(k, synth.C2_WIRE_BYTES)
            assert np.array_equal(h_out[:k * slot].reshape(k, slot)[:, :synth.C2_WIRE_BYTES], dev_out), "host path and resident path disagree"
            tail = h_out.reshape(n, slot)[-k:, :synth.C2_WIRE_BYTES]
            dev_tail = resp.out[(n - k) * synth.C2_WIRE_BYTES:n * synth.C2_WIRE_BYTES].cpu().numpy().reshape(k, synth.C2_WIRE_BYTES)
            assert np.array_equal(tail, dev_tail), "host path and resident path disagree"
        else:
            h_out = pinned_array(out_bytes + 4096)
            h_off = pinned_array(4 * (n + 1), np.uint32)
            h_meta = pinned_array(4 * n, np.uint32)
            for _ in range(args.warmup):
                got = eng.serve_host(hb, date, h_out, h_off, h_meta)
            assert got == out_bytes
            barrier()
            t0 = time.perf_counter()
            for _ in range(ksteps):
                eng.serve_host(hb, date, h_out, h_off, h_meta)
            barrier()
            dt = reduce_max(time.perf_counter() - t0)
            d2h = out_bytes + 4 * n + 4 * n + 8 * ((n + args.chunk - 1) // args.chunk)
            # the last host result must match the resident one byte for byte
            dev_out = resp.out[:out_bytes].cpu().numpy()
            assert np.array_equal(h_out[:out_bytes], dev_out), "host path and resident path disagree"
        barrier()
        floor = reduce_max(link_floor_ms(dev, int(h2d), int(d2h)))
        barrier()
        e2e = {"value": n * world * ksteps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": dt / ksteps * 1e3, "steps": ksteps, "chunk_requests": args.chunk, "layout": args.e2e_layout,
               "timing": "wall clock around the synchronous host-buffer calls, max over ranks",
               "link_floor_ms_per_step": floor,
               "link_floor": "the same H2D + D2H bytes per rank moved concurrently on all ranks with no kernel (pinned buffers, "
                             "max over ranks): what PCIe and host memory allow at this N",
               "frac_of_link_floor": floor / (dt / ksteps * 1e3)}

    # ---- CPU baseline beside it (rank 0, bounded sample of the same stream) ----
    cpu = None
    if rank == 0:
        from tests import oracle as O
        m = min(args.cpu_sample, n)
        sb = synth.config2_batch(m)
        ot = O.OracleTable(synth.config2_spec(S.FRAME_WIRE))
        cap = m * 640 + 4096
        o = np.zeros(cap, dtype=np.uint8)
        f = np.zeros(m + 1, dtype=np.uint32)
        mt = np.zeros(m, dtype=np.uint32)
        if world == 1:   # timed at N=1 only: at N>1 the other ranks' barrier spin shares the host's CPU quota
            reps = 4
            # the CPU arm gets every CPU the process started with, not just the GPU's NUMA node (the pthreads it starts
            # inherit this thread's affinity): the same footing as `--impl reference`
            cpus_bound = os.sched_getaffinity(0)
            os.sched_setaffinity(0, cpus_before_bind)
            cores, quota = pick_cpu_threads(lambda c: O.lib().orc_serve(
                ot._t, sb.desc.ctypes.data, sb.trace_ids.ctypes.data, sb.arena.ctypes.data, m, date, o.ctypes.data, cap,
                f.ctypes.data, mt.ctypes.data, c))
            t0 = time.perf_counter()
            for _ in range(reps):
                O.lib().orc_serve(ot._t, sb.desc.ctypes.data, sb.trace_ids.ctypes.data, sb.arena.ctypes.data, m, date,
                                  o.ctypes.data, cap, f.ctypes.data, mt.ctypes.data, cores)
            dtc = time.perf_counter() - t0
            cpu = {"value": m * reps / dtc, "unit": UNIT, "cores": cores, "kind": "port",
                   "cpu_quota": quota,
                   "sample": f"{reps} passes over the first {m} requests of the same stream, {cores} pthreads of "
                             f"{os.cpu_count()} logical CPUs (cgroup CPU quota: {quota if quota else 'none'}), in-memory, "
                             f"affinity: {len(cpus_before_bind)} CPUs"}
            os.sched_setaffinity(0, cpus_bound)
        # the sample doubles as a parity check of the bench's own output
        o1, f1, _ = ot.serve(sb.slice(0, 4096), date)
        g = resp.out[:4096 * synth.C2_WIRE_BYTES].cpu().numpy()
        assert np.array_equal(g, o1[:4096 * synth.C2_WIRE_BYTES]), "bench output differs from the oracle"

    # ---- the headline line is complete here; the sharded legs below can only add keys to it ----
    line = None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": workload_config(n, world, args),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": profiled_traffic(args.layout) if n == (1 << 20) else None, "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes,
                             "algorithmic_bytes_per_request": algo_bytes / n, "kernel_ms_per_launch": per_launch_ms,
                             "kernel": ("gofr::serve_slots_kernel_wide (4 CTAs/SM, 128 registers)" if eng.slot_ctas() == 4 else
                                        "gofr::serve_slots_kernel (5 CTAs/SM)") if args.layout == "slots" else "gofr::serve_kernel"},
                "other_layout": alt,
                "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
                "geometry": eng.geometry(), "numa": numa}
    printed = threading.Lock()

    def emit(extra):
        """Exactly one JSON line per job, whoever gets here first (the normal exit or the watchdog below)."""
        if not printed.acquire(blocking=False):
            return
        if rank == 0:
            print(json.dumps({**line, **extra}), flush=True)

    # ---- sharded legs of the other BASELINE configs (config 4 on 4 GPUs, config 5 on 8 GPUs) ----
    extras = {}
    watchdog = None
    if not args.no_extras and world in (4, 8):
        # A leg that stalls (one rank raising inside it leaves the others at a barrier) must not take the measured headline
        # with it: after --extras-timeout seconds every rank's watchdog ends the process, rank 0 printing the line first.
        def give_up():
            emit({"sharded_leg_error": "timed out after %d s; headline unaffected" % args.extras_timeout})
            sys.stdout.flush()
            os._exit(0)
        watchdog = threading.Timer(args.extras_timeout, give_up)
        watchdog.daemon = True
        watchdog.start()
    if not args.no_extras:
        # a leg that raises the same way on every rank (a programming error) must not take the headline line with it
        try:
            if world == 4:
                extras["config4_sharded"] = sharded_config4(eng_factory=lambda spec: Engine(Table(image=gd.broadcast_table_image(
                    Table(spec).serialize() if rank == 0 else None, rank, dev)), local), rank=rank, world=world, dev=dev,
                    barrier=barrier, reduce_max=reduce_max, steps=args.steps)
            if world == 8:
                extras["config5_sharded"] = sharded_config5(eng, rank, world, dev, barrier, reduce_max, args.steps)
        except Exception as ex:  # noqa: BLE001
            extras["sharded_leg_error"] = repr(ex)[:300]

    if watchdog is not None:
        watchdog.cancel()
    emit(extras)
    if world > 1:
        # the line is out; a rank that left a leg early (its own exception) must not wait forever for the others here
        bye = threading.Timer(60, lambda: os._exit(0))
        bye.daemon = True
        bye.start()
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
