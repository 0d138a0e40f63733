#!/usr/bin/env python
"""bench.py — xPNG encode/decode MPix/s on B200 (BASELINE.json metric), one JSON line.

Workload: BASELINE configs[2] — a fixed batch of F sintel-like 1920x1080 RGB frames (seeds 1000.., SURVEY.md §8(d);
F = 1000 unless --frames / XPNG_BENCH_FRAMES says otherwise), cut contiguously over the N ranks with
xpngb_shard_range (STRONG scaling: the batch is fixed, every rank codes its shard on its own GPU with no data-path
collective).  A "step" is one pass of the hot path over the batch:

    for level in (1, 2):  encode shard  ->  size/offset gather over all ranks (C, shared memory)  ->  decode shard

  value : whole-job MPix/s = 4 codec calls x batch pixels / step time, pixels and files resident in HBM, CUDA events
          on the codec's stream, max over ranks.  Level 7 (a device copy) is measured on its own and reported in
          `breakdown`, not folded into `value`.
  e2e   : the same step through the C ABI with pinned HOST buffers (H2D and D2H inside the timed region).
  breakdown : per level and direction ms, MPix/s and algorithmic GB/s; level 7; a single 3840x2160 frame (configs[1])
          as the `latency` record; `e2e_file`: the repo's own xpng_store_T / xpng_load_T through tmpfs.
  roofline / cpu_baseline: see DESIGN.md "Measurement".

--impl reference times the unmodified reference (oracle/_ref, built from /root/reference by oracle/Makefile) on the
host cores with all the threads it spawns by itself (T = 0 -> nproc), on a bounded sample of the same frames, through
its own file API on tmpfs.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA initialises (see xpng_b200/__init__.py)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
FW, FH = 1920, 1080
SEED0 = 1000
LEVELS = (1, 2)
METRIC = "xpng encode+decode MPix/s at levels -1/-2 over a 1080p frame batch"
REF_SAMPLE = 64
DUMP_FILE_BYTES = 1 << 22      # --dump-outputs: sampled file bytes per level (16 MiB as float32)
DUMP_PIXEL_BYTES = 1 << 21     # --dump-outputs: sampled decoded bytes per level (8 MiB as float32)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bind_near_gpu(index):
    """Run this thread (and the threads it starts, and the pinned host memory it allocates: first touch) on the CPUs of the
    GPU's NUMA node; a host buffer on the far socket costs a third of the PCIe rate.  Returns (record for the JSON line, the
    affinity to restore before the CPU legs)."""
    orig = os.sched_getaffinity(0)
    try:
        import pynvml as N
        N.nvmlInit()
        bus = N.nvmlDeviceGetPciInfo(N.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        dom, rest = bus.split(":", 1)
        dev = f"/sys/bus/pci/devices/{dom[-4:]}:{rest}"
        node = int(open(dev + "/numa_node").read())
        cpus = set()
        for part in open(dev + "/local_cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= orig
        if node >= 0 and cpus and cpus != orig:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus), "of": len(orig)}, orig
        return {"numa_node": node, "cpus": len(orig), "of": len(orig)}, orig
    except Exception as e:
        return {"numa_node": None, "note": f"not bound ({type(e).__name__})"}, orig


def pcie_probe(torch, dev, h_buf, d_buf, nbytes):
    """What the box gives between pinned host memory and the GPU: GB/s up, down, and both at once (two streams)."""
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    h2 = torch.empty(nbytes, dtype=torch.uint8).pin_memory(); d2 = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    def run(up, down):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        if up:
            with torch.cuda.stream(s1): d_buf[:nbytes].copy_(h_buf[:nbytes], non_blocking=True)
        if down:
            with torch.cuda.stream(s2): h2.copy_(d2, non_blocking=True)
        torch.cuda.synchronize(); return time.perf_counter() - t0
    run(1, 1)
    up = min(run(1, 0) for _ in range(2)); down = min(run(0, 1) for _ in range(2)); both = min(run(1, 1) for _ in range(2))
    return {"h2d_GB_s": round(nbytes / 1e9 / up, 1), "d2h_GB_s": round(nbytes / 1e9 / down, 1), "duplex_GB_s": round(2 * nbytes / 1e9 / both, 1)}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def _run_nvml(self):
        """Fast path: NVML in-process (10 ms period); returns False when NVML is unavailable."""
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.index)
            mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        except Exception:
            return False
        while not self._stop_evt.is_set():
            try:
                sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
                r = int(get_reasons(h))
                self.rows.append([str(self.index), str(sm), str(mx)] + ["Active" if r & bits[k] else "Not Active"
                                                                         for k in ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")])
            except Exception:
                pass
            self._stop_evt.wait(0.01)
        return True

    def run(self):
        if self._run_nvml():
            return
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(int(r[1]) for r in self.rows if r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if r[2].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ reference arm

def _quiet_call(fn, *a):
    """Run fn with fd 1 pointed at /dev/null (the reference prints a MPx/s line per call, NCCL its version)."""
    sys.stdout.flush()
    saved = os.dup(1)
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 1)
    try:
        return fn(*a)
    finally:
        os.dup2(saved, 1)
        os.close(saved)
        os.close(devnull)


class _Xpng(C.Structure):
    _fields_ = [("p", C.c_void_p), ("w", C.c_uint64), ("h", C.c_uint64), ("s", C.c_uint64), ("A", C.c_bool)]


def _tmpdir():
    return "/dev/shm" if os.path.isdir("/dev/shm") else "/tmp"


def file_api_steps(L, frames, steps, warmup, tag, callers=1):
    """K steps of the file-at-a-time API (xpng_store_T / xpng_load_T, T = 0) over `frames` at levels 1 and 2, files on tmpfs.
    `L` is a CDLL exporting the reference's entry points (the reference itself or this repo's drop-in).
    callers > 1: the frames of a level are handed to that many host threads (the API is re-entrant; one frame per call either way).
    Returns (seconds per step, {call: seconds per step})."""
    L.xpng_store_T.restype = C.c_bool
    L.xpng_store_T.argtypes = [C.c_uint64, C.c_uint64, C.POINTER(_Xpng), C.c_char_p]
    L.xpng_load_T.restype = C.c_bool
    L.xpng_load_T.argtypes = [C.c_uint64, C.c_char_p, C.POINTER(_Xpng)]
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    pms = [_Xpng(f.ctypes.data, f.shape[1], f.shape[0], f.size, f.shape[2] == 4) for f in frames]
    paths = [os.path.join(_tmpdir(), f"_xpng_{tag}_{os.getpid()}_{i}.xpng").encode() for i in range(len(frames))]
    per_call = {}

    tp = ThreadPoolExecutor(callers) if callers > 1 else None
    each = (lambda fn, items: list(tp.map(fn, items))) if tp else (lambda fn, items: [fn(it) for it in items])

    def store(lv):
        def one(k):
            assert not L.xpng_store_T(0, lv, C.byref(pms[k]), paths[k])
        return one

    def load(k):
        out = _Xpng()
        assert not L.xpng_load_T(0, paths[k], C.byref(out))
        libc.free(C.c_void_p(out.p))

    def step(rec):
        for lv in LEVELS:
            t0 = time.perf_counter()
            each(store(lv), range(len(pms)))
            t1 = time.perf_counter()
            each(load, range(len(pms)))
            t2 = time.perf_counter()
            if rec:
                per_call[f"enc{lv}"] = per_call.get(f"enc{lv}", 0.0) + (t1 - t0)
                per_call[f"dec{lv}"] = per_call.get(f"dec{lv}", 0.0) + (t2 - t1)
    times = []
    try:
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            _quiet_call(step, i >= warmup)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    finally:
        if tp:
            tp.shutdown()
        for p in paths:
            if os.path.exists(p):
                os.remove(p)
    return sum(times) / len(times), {k: v / steps for k, v in per_call.items()}


def reference_steps(frames, steps, warmup):
    """CPU baseline on `frames`: the unmodified reference when it travelled (oracle/_ref), else the oracle port."""
    ref_so = os.path.join(ROOT, "oracle", "_ref", "libxpng_ref.so")
    if os.path.exists(ref_so):
        per_step, calls = file_api_steps(C.CDLL(ref_so), frames, steps, warmup, "ref")
        return per_step, calls, "reference", os.cpu_count(), "xpng_store_T/xpng_load_T (T=0: all host cores), files on tmpfs"
    from oracle import pyoracle as po
    calls = {}
    t_all = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        for lv in LEVELS:
            ta = time.perf_counter()
            files = [po.encode(lv, f) for f in frames]
            tb = time.perf_counter()
            for f in files:
                po.decode(f)
            tc = time.perf_counter()
            if i >= warmup:
                calls[f"enc{lv}"] = calls.get(f"enc{lv}", 0.0) + (tb - ta) / steps
                calls[f"dec{lv}"] = calls.get(f"dec{lv}", 0.0) + (tc - tb) / steps
        if i >= warmup:
            t_all.append(time.perf_counter() - t0)
    return sum(t_all) / len(t_all), calls, "port", 1, "single-threaded oracle port, in memory"


def call_table(calls, npx_total):
    return {k: {"ms": round(v * 1e3, 3), "MPix_s": round(npx_total / 1e6 / v, 1)} for k, v in sorted(calls.items())}


def run_reference(args, rank, world):
    if rank != 0:
        return
    from xpng_b200 import synth
    nf = min(args.frames, REF_SAMPLE)
    frames = synth.sintel_batch(range(SEED0, SEED0 + nf))
    steps = args.steps
    per_step, calls, kind, cores, how = reference_steps(frames, steps, args.warmup)
    npx = nf * FW * FH
    value = 4 * npx / 1e6 / per_step
    sample = (f"first {nf} of the {args.frames} frames of the same batch (config is the GPU arm's; the CPU arm codes a bounded sample), "
              f"levels 1 and 2, encode then decode of every frame per level, {how}")
    line = {"metric": METRIC, "value": round(value, 2), "unit": "MPix/s", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
            "ms_per_step": round(per_step * 1e3, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "impl": "reference",
            "config": dict(workload_config(args.frames, world), parts_per_level=max(1, args.parts), schedule=args.schedule, e2e_schedule=args.e2e_schedule),
            "cpu_baseline": {"value": round(value, 2), "unit": "MPix/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": round(value, 2), "unit": "MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "breakdown": call_table(calls, npx)}
    print(json.dumps(line), flush=True)


def _sample_positions(n, k, seed):
    """Every position below n when n <= k, else k fixed, seeded positions in increasing order."""
    return np.arange(n, dtype=np.int64) if n <= k else np.sort(np.random.default_rng(seed).integers(0, n, k, dtype=np.int64))


def dump_outputs(out_dir, files, back, offs, sizes, npx_bytes):
    """Write what a step handed back, per level L, as .npy files under out_dir (about 50 MB in all):
    L<L>_sizes / L<L>_offsets (float64): every file's size and its offset in the file arena;
    L<L>_file_bytes (float32): the files of all frames concatenated in frame order, every byte or a fixed seeded sample;
    L<L>_decoded_pixels (float32): the decoded pixel arena, every byte or a fixed seeded sample.
    The inputs depend on the arguments only, so two builds run with the same arguments can be compared file for file."""
    import torch
    os.makedirs(out_dir, exist_ok=True)

    def take(t, idx):
        return t[torch.from_numpy(idx).to(t.device)].float().cpu().numpy()
    for lv in LEVELS:
        sz, of = np.asarray(sizes[lv], np.int64), np.asarray(offs[lv], np.int64)
        starts = np.cumsum(sz) - sz                              # where each file begins in the concatenation
        pos = _sample_positions(int(sz.sum()), DUMP_FILE_BYTES, lv)
        k = np.searchsorted(starts, pos, side="right") - 1
        out = {"sizes": sz.astype(np.float64), "offsets": of.astype(np.float64),
               "file_bytes": take(files[lv], of[k] + (pos - starts[k])),
               "decoded_pixels": take(back[lv], _sample_positions(npx_bytes, DUMP_PIXEL_BYTES, 100 + lv))}
        for name, a in out.items():
            np.save(os.path.join(out_dir, f"L{lv}_{name}.npy"), a)


def workload_config(frames, world):
    cfg = {"workload": f"configs[2]: {frames} sintel-like 1920x1080 RGB frames (seeds {SEED0}..{SEED0 + frames - 1}), levels -1/-2, "
                       "encode + size/offset gather + decode per level",
           "frames": frames, "tiles_per_frame": 8,
           "l2": "no flush needed: a rank's pixels, files and scratch are far larger than the 126 MB L2 (>= 0.7 GB per rank at N = 8)",
           "parallelism": f"frames sharded contiguously over {world} GPU(s) (xpngb_shard_range), no data-path collective; "
                          "one shared-memory size gather per level (xpngb_gather_sizes, C, no NCCL)"}
    return cfg


# ------------------------------------------------------------------------------------------------ our arm

def run_ours(args, rank, world, local_rank):
    import torch
    import xpng_b200
    from xpng_b200 import shard, synth
    from oracle import pyoracle as po

    dist = None
    if world > 1:
        import torch.distributed as dist                      # the clock only: barrier + max over ranks
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        _quiet_call(lambda: (dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank)), dist.barrier()))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity, all_cpus = bind_near_gpu(local_rank)          # before any pinned allocation or worker thread
    lib = xpng_b200.lib()
    # A step is a set of JOBS: (level, part of the shard) -> encode, [size/offset gather once the level is encoded], decode.
    # Every job has its own codec context and host thread, so the serial-chain phases of one job overlap the
    # data-parallel phases of the others on the device, and with host buffers the pixel uploads of one job's encode
    # run next to the pixel downloads of another job's decode (both PCIe directions busy).
    F = args.frames
    lo, hi = shard.shard_range(F, rank, world)
    n = hi - lo
    PARTS = max(1, min(args.parts, n if n else 1))
    part_rng = [shard.shard_range(n, p, PARTS) for p in range(PARTS)]          # frame ranges of the parts inside the shard
    JOBS = [(lv, p) for lv in LEVELS for p in range(PARTS)]
    cds = {j: xpng_b200.Codec(local_rank) for j in JOBS}
    cd = cds[JOBS[0]]
    stream = torch.cuda.ExternalStream(cd.stream, device=dev)
    gtag = f"bench{os.environ.get('MASTER_PORT', '0')}_{os.environ.get('TORCHELASTIC_RUN_ID', os.getppid() if world > 1 else os.getpid())}"
    gathers = {lv: shard.Gather(f"{gtag}_L{lv}", rank, world, F) for lv in LEVELS}
    npx_frame = FW * FH
    FRAME_B = npx_frame * 3                      # 6220800: a multiple of 16, frame k of the shard sits at k * FRAME_B
    FILE_B = (8 + FRAME_B + 15) & ~15            # xpngb_encode_bound of one frame: part p's files start at a * FILE_B
    shapes = [(FH, FW, 3)] * n
    descs0, total = xpng_b200.Codec.layout(shapes)
    cap = int(lib.xpngb_encode_bound(descs0, n)) if n else 16
    assert total == n * FRAME_B and (cap == n * FILE_B or not n)
    # ---- frames of this rank's shard, generated straight into pinned host memory, then uploaded
    h_px = torch.empty(max(total, 16) + 64, dtype=torch.uint8).pin_memory()
    frames_sample = {}
    if n:
        hv = h_px.numpy()
        sample_idx = sorted({0, n // 3, (2 * n) // 3, n - 1})
        for k0 in range(0, n, 64):
            part = synth.sintel_batch(range(SEED0 + lo + k0, SEED0 + lo + min(k0 + 64, n)))
            for k, f in enumerate(part):
                o = descs0[k0 + k].offset
                hv[o:o + f.size] = f.reshape(-1)
                if k0 + k in sample_idx:
                    frames_sample[k0 + k] = f
    d_px = h_px.to(dev)
    d_files = {lv: torch.zeros(cap + 64, dtype=torch.uint8, device=dev) for lv in LEVELS}
    d_back = {lv: torch.zeros(max(total, 16) + 64, dtype=torch.uint8, device=dev) for lv in LEVELS}
    state = {"launches": 0, "calls": {}, "sizes": {lv: [0] * n for lv in LEVELS}, "offs": {lv: [0] * n for lv in LEVELS}, "sha": {}, "table_sha": None}
    pool = ThreadPoolExecutor(len(JOBS))
    lock = threading.Lock()

    def part_descs(m, zero_dims=False):
        d = xpng_b200.Codec.layout(shapes[:m])[0]
        if zero_dims:
            for x in d:
                x.w = x.h = 0
        return d

    def job(i, px, files, back, on_dev, rec, chained, evs, left):
        lv, p = JOBS[i]
        c = cds[JOBS[i]]
        a, b = part_rng[p]
        m = b - a
        if chained and i > 0:
            evs[i - 1].wait()                        # my encode starts when the previous job has encoded
        t0 = time.perf_counter()
        # the part's region of the level's file arena: device arenas hold the bound, the pinned host arenas what the parts need
        fbase, fcap = (a * FILE_B, m * FILE_B) if on_dev else state["hregion"][lv][p]
        if m:
            offs, sz = c.encode_raw(lv, part_descs(m), m, px.data_ptr() + a * FRAME_B, m * FRAME_B, on_dev,
                                    files[lv].data_ptr() + fbase, fcap, on_dev)
            launches = c.last_launches
            state["sizes"][lv][a:b] = [int(sz[k]) for k in range(m)]
            state["offs"][lv][a:b] = [fbase + int(offs[k]) for k in range(m)]
        else:
            offs, sz, launches = (C.c_uint64 * 1)(), (C.c_uint64 * 1)(), 0
        t1 = time.perf_counter()
        evs[i].set()
        with lock:
            left[lv] -= 1
            last = left[lv] == 0
        if last:                                     # the level is encoded: the one exchange between ranks
            g_offs, g_sizes = gathers[lv].sizes(F, list(state["sizes"][lv]))
            h = hashlib.sha256()
            h.update(np.asarray(g_sizes, dtype=np.uint64).tobytes()); h.update(np.asarray(g_offs, dtype=np.uint64).tobytes())
            state["sha"][lv] = h.hexdigest()
        t2 = time.perf_counter()
        if m:
            c.decode_raw(part_descs(m, True), m, files[lv].data_ptr() + fbase, fcap, on_dev, offs, sz,
                         back[lv].data_ptr() + a * FRAME_B, m * FRAME_B, on_dev)
            launches += c.last_launches
        t3 = time.perf_counter()
        with lock:
            state["launches"] += launches
            if rec:
                cc = state["calls"]
                cc[f"enc{lv}"] = cc.get(f"enc{lv}", 0.0) + (t1 - t0); cc[f"dec{lv}"] = cc.get(f"dec{lv}", 0.0) + (t3 - t2)
                if last:
                    cc[f"gather{lv}"] = cc.get(f"gather{lv}", 0.0) + (t2 - t1)

    def step(px, files, back, on_dev, rec, schedule="concurrent"):
        evs = [threading.Event() for _ in JOBS]
        left = {lv: PARTS for lv in LEVELS}
        if schedule == "sequential":
            for i in range(len(JOBS)):
                job(i, px, files, back, on_dev, rec, False, evs, left)
        else:
            for fu in [pool.submit(job, i, px, files, back, on_dev, rec, schedule == "chained", evs, left) for i in range(len(JOBS))]:
                fu.result()
        state["table_sha"] = hashlib.sha256("".join(state["sha"][lv] for lv in LEVELS).encode()).hexdigest()[:16]

    def timed(px, files, back, on_dev, steps, warmup, schedule="concurrent"):
        for _ in range(warmup):
            step(px, files, back, on_dev, False, schedule)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        state["launches"] = 0; state["calls"] = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(steps):
            step(px, files, back, on_dev, True, schedule)   # every call returns with its device work done: e1 closes the region
        e1.record(stream)
        e1.synchronize()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.barrier()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), {k: v / steps for k, v in state["calls"].items()}

    # ---- parity gate before any timing counts (BASELINE.md §2): sampled frames byte for byte against the oracle,
    # every decoded pixel of the shard against the input
    step(d_px, d_files, d_back, 1, False)
    for lv in LEVELS:
        for k, f in frames_sample.items():
            o, s = state["offs"][lv][k], state["sizes"][lv][k]
            got = d_files[lv][o:o + s].cpu().numpy().tobytes()
            assert got == po.encode(lv, f), f"rank {rank} level {lv} frame {lo + k}: bytes differ from the oracle"
        if n:
            assert torch.equal(d_back[lv][:total], d_px[:total]), f"rank {rank} level {lv}: decoded pixels differ"
    xpng_bytes = {lv: sum(state["sizes"][lv]) for lv in LEVELS}

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_dev, calls_conc = timed(d_px, d_files, d_back, 1, args.steps, args.warmup, args.schedule)
    n_launch = state["launches"]
    clocks = sampler.stop()
    for lv in LEVELS:
        if n:
            assert torch.equal(d_back[lv][:total], d_px[:total]), f"rank {rank} level {lv}: decoded pixels differ after the timed steps"
    if args.dump_outputs and rank == 0:                       # before the legs below overwrite the arenas
        dump_outputs(args.dump_outputs, d_files, d_back, state["offs"], state["sizes"], total)
    # the same step with the two level jobs one after the other: per-call device-resident times for the breakdown
    ms_seq, calls_dev = timed(d_px, d_files, d_back, 1, 2, 1, "sequential")
    table_sha = state["table_sha"]
    dev_offs = {lv: list(state["offs"][lv]) for lv in LEVELS}     # the device arena's layout (the host leg packs differently)
    dev_sizes = {lv: list(state["sizes"][lv]) for lv in LEVELS}
    # ---- end to end: pinned host buffers through the same C ABI calls
    state["hregion"] = {}
    h_files = {}
    for lv in LEVELS:      # host arenas: one region per part, sized from the sizes the device leg produced (+5 %)
        regs, base = [], 0
        for (a, b) in part_rng:
            need = (int(sum(dev_sizes[lv][a:b]) * 1.05) + (1 << 20) + 15) & ~15
            regs.append((base, need)); base += need
        state["hregion"][lv] = regs
        h_files[lv] = torch.empty(max(base, 16) + 64, dtype=torch.uint8).pin_memory()
    h_back = {lv: torch.empty(max(total, 16) + 64, dtype=torch.uint8).pin_memory() for lv in LEVELS}
    pcie = pcie_probe(torch, dev, h_px, d_px, min(total, 1 << 30)) if n else None
    e2e_steps = max(1, min(args.steps, 3))
    ms_e2e, calls_e2e = timed(h_px, h_files, h_back, 0, e2e_steps, 1, args.e2e_schedule)
    if n:
        for lv in LEVELS:
            assert np.array_equal(h_back[lv].numpy()[:total], h_px.numpy()[:total]), f"e2e level {lv}: decoded pixels differ"

    npx_total = F * npx_frame
    value = 4 * npx_total / 1e6 / (ms_dev / args.steps / 1e3)
    e2e = 4 * npx_total / 1e6 / (ms_e2e / e2e_steps / 1e3)
    raw_shard = n * npx_frame * 3
    # all ranks: the shard's bytes, summed by the driver's view below (rank 0 reports the whole job: every shard is the same size +-1 frame)
    sums = torch.tensor([raw_shard, xpng_bytes[1], xpng_bytes[2]], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    raw_all, x1_all, x2_all = (int(v) for v in sums.tolist())
    if rank != 0:
        for g in gathers.values():
            g.close()
        return
    h2d = 2 * raw_all + x1_all + x2_all      # encodes upload the pixels, decodes upload the files
    d2h = x1_all + x2_all + 2 * raw_all
    alg = {1: raw_all + x1_all, 2: raw_all + x2_all}
    peak, peak_src = peaks()

    def table(calls):
        out = {}
        for k, v in sorted(calls.items()):
            if k.startswith("gather"):
                out[k] = {"ms": round(v * 1e3, 3)}
            else:
                lv = int(k[-1])
                out[k] = {"ms": round(v * 1e3, 3), "MPix_s": round(npx_total / 1e6 / v, 1), "GB_s": round(alg[lv] / 1e9 / v, 1),
                          "hbm_frac": round(alg[lv] / 1e9 / v / (peak * world), 4)}
        return out
    breakdown = {"device_sequential": table(calls_dev), "device_sequential_ms_per_step": round(ms_seq / 2, 3),
                 "device_concurrent_levels": table(calls_conc), "e2e": table(calls_e2e),
                 "note": "value / e2e: a step's levels x parts jobs run on one codec context and host thread each (config.schedule / e2e_schedule); "
                         "device_sequential: the same calls one at a time (per-call times without overlap, summed over the parts)"}

    # ---- level 7 on its own (stored files: a device copy)
    if n:
        t7 = {}
        for _ in range(3):
            t0 = time.perf_counter()
            offs7, sz7 = cd.encode_raw(7, part_descs(n), n, d_px.data_ptr(), total, 1, d_files[1].data_ptr(), cap, 1)
            t1 = time.perf_counter()
            cd.decode_raw(part_descs(n, True), n, d_files[1].data_ptr(), cap, 1, offs7, sz7, d_back[1].data_ptr(), total, 1)
            t2 = time.perf_counter()
            t7["enc7"] = min(t7.get("enc7", 1e9), t1 - t0); t7["dec7"] = min(t7.get("dec7", 1e9), t2 - t1)
        npx_shard = n * npx_frame
        breakdown["level7_rank0_shard"] = {k: {"ms": round(v * 1e3, 3), "MPix_s": round(npx_shard / 1e6 / v, 1), "GB_s": round(2 * raw_shard / 1e9 / v, 1)}
                                           for k, v in t7.items()}

    # ---- per-kernel view of one step (serialised profiling pass, outside the timed region) and the dominant kernel
    per_kernel = {}
    for lv in LEVELS:
        prof_offs = prof_sz = None
        for what in ("enc", "dec"):
            cd.profile(True)
            if what == "enc":
                prof_offs, prof_sz = cd.encode_raw(lv, part_descs(n), n, d_px.data_ptr(), total, 1, d_files[lv].data_ptr(), cap, 1)
            else:
                cd.decode_raw(part_descs(n, True), n, d_files[lv].data_ptr(), cap, 1, prof_offs, prof_sz, d_back[lv].data_ptr(), total, 1)
            for k, (ms, cnt) in cd.profile_report().items():
                per_kernel[f"L{lv}.{what}.{k}"] = (ms, cnt, lv)
            cd.profile(False)
    top_name, (top_ms, top_cnt, top_lv) = max(per_kernel.items(), key=lambda kv: kv[1][0])
    alg_shard = raw_shard + xpng_bytes[top_lv]              # algorithmic bytes of the call the kernel belongs to (rank 0's shard)
    achieved = alg_shard / 1e9 / (top_ms / 1e3)
    traffic, traffic_src = None, None
    try:   # DRAM bytes per pixel of that kernel from the committed ncu --set full capture, scaled to this launch
        tj = json.load(open(os.path.join(ROOT, "profiles", "r03_traffic.json")))
        base = top_name.split(".")[-1]
        for name, rec in tj.items():
            if name == base:
                traffic = int(rec["dram_bytes_per_pixel"] * n * npx_frame / top_cnt); traffic_src = "profiles/" + rec["report"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": top_name, "launches": top_cnt, "kernel_ms_per_launch": round(top_ms / top_cnt, 4),
                "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 5),
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_shard // top_cnt,
                "note": "achieved = (raw + xpng bytes of the call's shard) / (sum of the kernel's launch durations in that call), CUDA events per launch "
                        "on the launching stream (xpngb_profile, serialised pass after the timed region)"}
    breakdown["step_algorithmic_GB_s"] = round(2 * (alg[1] + alg[2]) / 1e9 / (ms_dev / args.steps / 1e3), 1)
    breakdown["step_hbm_frac"] = round(2 * (alg[1] + alg[2]) / 1e9 / (ms_dev / args.steps / 1e3) / (peak * world), 4)
    breakdown["kernels_ms_rank0"] = {k: round(v[0], 3) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1][0])[:12]}

    # ---- latency record: one 3840x2160 frame (BASELINE configs[1]) per call
    frame4k = synth.rgb(2160, 3840, 1)
    d4, tot4 = xpng_b200.Codec.layout([frame4k.shape])
    cap4 = int(lib.xpngb_encode_bound(d4, 1))
    p4 = torch.from_numpy(frame4k.reshape(-1)).to(dev); p4 = torch.cat([p4, torch.zeros(64, dtype=torch.uint8, device=dev)])
    f4 = torch.zeros(cap4 + 64, dtype=torch.uint8, device=dev); b4 = torch.zeros(tot4 + 64, dtype=torch.uint8, device=dev)
    lat = {}
    for lv in (1, 2, 7):
        be = bd = 1e9
        for _ in range(4):
            d = xpng_b200.Codec.layout([frame4k.shape])[0]
            t0 = time.perf_counter()
            o4, s4 = cd.encode_raw(lv, d, 1, p4.data_ptr(), tot4, 1, f4.data_ptr(), cap4, 1)
            t1 = time.perf_counter()
            d = xpng_b200.Codec.layout([frame4k.shape])[0]; d[0].w = d[0].h = 0
            cd.decode_raw(d, 1, f4.data_ptr(), cap4, 1, o4, s4, b4.data_ptr(), tot4, 1)
            t2 = time.perf_counter()
            be = min(be, t1 - t0); bd = min(bd, t2 - t1)
        assert torch.equal(b4[:tot4], p4[:tot4])
        lat[f"enc{lv}_ms"] = round(be * 1e3, 3); lat[f"dec{lv}_ms"] = round(bd * 1e3, 3)
    breakdown["latency_4k_frame"] = lat

    # ---- the repo's own file API (xpng_store_T / xpng_load_T through tmpfs), like the reference arm does it
    breakdown["pcie_probe"] = pcie
    breakdown["host_affinity"] = affinity
    os.sched_setaffinity(0, all_cpus)                         # the CPU legs below use every host core, like the reference arm
    cpu = None
    if world == 1:
        sample = synth.sintel_batch(range(SEED0, SEED0 + min(F, 16)))
        per_step, calls = file_api_steps(C.CDLL(xpng_b200.lib_path()), sample, 2, 1, "ours")
        breakdown["e2e_file"] = {"MPix_s": round(4 * len(sample) * npx_frame / 1e6 / per_step, 1), "frames": len(sample),
                                 "how": "this library's xpng_store_T/xpng_load_T, one frame per call, files on tmpfs (the reference arm's own method)",
                                 "calls": call_table(calls, len(sample) * npx_frame)}
        try:    # the same calls from eight host threads at once: what a multi-threaded caller of the re-entrant API sees
            per_step8, calls8 = file_api_steps(C.CDLL(xpng_b200.lib_path()), sample, 2, 1, "ours8", callers=8)
            breakdown["e2e_file_8_callers"] = {"MPix_s": round(4 * len(sample) * npx_frame / 1e6 / per_step8, 1), "frames": len(sample),
                                               "how": "as e2e_file, the frames of a level handed to 8 host threads (one frame per call, contexts from the library's pool)",
                                               "calls": call_table(calls8, len(sample) * npx_frame)}
        except Exception as e:
            breakdown["e2e_file_8_callers"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
        if not args.no_cpu_baseline:
            nref = min(F, 32)
            ref_frames = synth.sintel_batch(range(SEED0, SEED0 + nref))
            per_step, calls, kind, cores, how = reference_steps(ref_frames, 2, 1)
            cpu = {"value": round(4 * nref * npx_frame / 1e6 / per_step, 2), "unit": "MPix/s", "cores": cores, "kind": kind,
                   "sample": f"first {nref} frames of the batch, levels 1 and 2, encode then decode per level, {how}; 2 steps after 1 warm-up",
                   "calls": call_table(calls, nref * npx_frame)}

    line = {"metric": METRIC, "value": round(value, 2), "unit": "MPix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_dev / args.steps, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic", "config": dict(workload_config(F, world), parts_per_level=PARTS, schedule=args.schedule, e2e_schedule=args.e2e_schedule),
            "e2e": {"value": round(e2e, 2), "unit": "MPix/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": round(ms_e2e / e2e_steps, 4), "steps": e2e_steps},
            "gpu_launches": n_launch, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "xpng_bytes": {"level1": x1_all, "level2": x2_all, "raw": raw_all}, "sizes_sha": table_sha, "breakdown": breakdown}
    print(json.dumps(line), flush=True)
    for g in gathers.values():
        g.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=int(os.environ.get("XPNG_BENCH_FRAMES", "1000")))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parts", type=int, default=int(os.environ.get("XPNG_BENCH_PARTS", "1")),
                    help="parts a rank's shard is cut into per level; a step runs levels x parts jobs (encode -> decode), one context each "
                         "(measured: 2 parts cost 28 %% device-resident, calls of 500 frames take almost as long as calls of 1000; 5 %% better end to end)")
    ap.add_argument("--schedule", default=os.environ.get("XPNG_BENCH_SCHEDULE", "concurrent"), choices=["concurrent", "chained", "sequential"],
                    help="device-resident leg: all jobs at once / each job's encode starts when the previous job has encoded / one job at a time")
    ap.add_argument("--e2e-schedule", default=os.environ.get("XPNG_BENCH_E2E_SCHEDULE", "chained"), choices=["concurrent", "chained", "sequential"],
                    help="host-buffer leg (chained keeps both PCIe directions busy: one job's decode downloads next to the next job's encode uploads)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (per level: file sizes and offsets, a fixed sample of "
                         "the file bytes and of the decoded pixels; rank 0's shard) as DIR/<name>.npy, float32 / float64, about 50 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what this library computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
