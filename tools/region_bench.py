#!/usr/bin/env python
"""Region decode against full decode on the GPU; one JSON line to profiles/region_bench_<tag>.json.

  A  batch: the bench.py workload (1000 sintel-like 1080p frames, seeds 1000..1999, files in device memory), levels 1
     and 2, one seeded 224 x 224 crop per frame: ms per xpngb_decode_region call against xpngb_decode of the same files,
     and the tiles each decodes (xpngb_region_tiles).
  B  single images: rgba_8192_s2 and a 4K RGB frame (rgb_4k_s1), crops of 256^2, 1024^2, a 2 x 2-tile union and the full
     image, with device-resident and with host buffers, against a full decode.
  C  k_crop_rows: GB/s over the bytes it reads and writes, from the per-kernel profile (xpngb_profile).

Every crop is compared with the full decode of the same file before anything is timed.  A timing is 3 warm-up calls and
then `--reps` calls, each ending in a device synchronise (the C calls return after one); median and minimum are reported.
Usage: python tools/region_bench.py [--frames 1000] [--reps 7] [--tag b200]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import xpng_b200  # noqa: E402
from xpng_b200 import synth  # noqa: E402
from xpng_b200.codec import _Image, rects  # noqa: E402
from conftest import make_case, manifest  # noqa: E402
from oracle import pyoracle as po  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "sm_clock_max": clock}


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": round(float(np.median(ts)), 3), "min_ms": round(float(np.min(ts)), 3)}


class Batch:
    """n files packed at 16-byte offsets, on the host and (copied once) on the device; output layouts for full and crops."""

    def __init__(self, files):
        self.n = n = len(files)
        self.foffs, self.fsizes = (C.c_uint64 * n)(), (C.c_uint64 * n)()
        off = 0
        for i, f in enumerate(files):
            self.foffs[i], self.fsizes[i] = off, len(f)
            off += (len(f) + 15) & ~15
        self.fsize = off
        self.pinned = torch.zeros(off + 64, dtype=torch.uint8).pin_memory()
        self.host = self.pinned.numpy()
        for i, f in enumerate(files):
            self.host[self.foffs[i]: self.foffs[i] + len(f)] = np.frombuffer(f, np.uint8)
        self.dev = self.pinned.cuda()
        self.hdr = []
        for i, f in enumerate(files):
            d = _Image()
            xpng_b200.lib().xpngb_peek(np.frombuffer(f[:8], np.uint8).ctypes.data, 8, C.byref(d))
            self.hdr.append((int(d.w), int(d.h), 3 + int(d.A)))

    def descs(self, boxes=None):
        arr, off = (_Image * self.n)(), 0
        for i, (w, h, c) in enumerate(self.hdr):
            arr[i].offset = off
            bw, bh = (w, h) if boxes is None else boxes[i][2:]
            off += (bw * bh * c + 15) & ~15
        return arr, off


def run_pair(cd, B, boxes, out_dev, files_dev, reps):
    """(full decode timing, region timing, crops) for one batch; crops checked against the full decode first."""
    fd, ftotal = B.descs()
    rd, rtotal = B.descs(boxes)
    ra = rects(boxes)
    if out_dev:
        fout = torch.empty(ftotal + 64, dtype=torch.uint8, device="cuda"); rout = torch.empty(rtotal + 64, dtype=torch.uint8, device="cuda")
        fptr, rptr = fout.data_ptr(), rout.data_ptr()
    else:
        fout = torch.empty(ftotal + 64, dtype=torch.uint8).pin_memory(); rout = torch.empty(rtotal + 64, dtype=torch.uint8).pin_memory()
        fptr, rptr = fout.data_ptr(), rout.data_ptr()
    fptr_files = B.dev.data_ptr() if files_dev else B.host.ctypes.data

    def full():
        cd.decode_raw(fd, B.n, fptr_files, B.fsize, int(files_dev), B.foffs, B.fsizes, fptr, ftotal, int(out_dev))

    def region():
        cd.decode_region_raw(rd, ra, B.n, fptr_files, B.fsize, int(files_dev), B.foffs, B.fsizes, rptr, rtotal, int(out_dev))

    full(); region(); torch.cuda.synchronize()
    fh, rh = fout.cpu().numpy(), rout.cpu().numpy()
    for i, (x, y, w, h) in enumerate(boxes):
        W, H, c = B.hdr[i]
        img = fh[fd[i].offset: fd[i].offset + W * H * c].reshape(H, W, c)
        crop = rh[rd[i].offset: rd[i].offset + w * h * c].reshape(h, w, c)
        if not np.array_equal(crop, img[y: y + h, x: x + w]):
            raise SystemExit(f"parity: entry {i} rect {(x, y, w, h)} differs from the full decode")
    tf = timed(full, reps); tf["kernel_ms"] = round(cd.last_kernel_ms, 3)
    tr = timed(region, reps); tr["kernel_ms"] = round(cd.last_kernel_ms, 3)
    return tf, tr


def tiles(B, boxes):
    full = sum(xpng_b200.region_tiles(w, h, (0, 0, w, h))[0] for w, h, _ in B.hdr)
    sel = sum(xpng_b200.region_tiles(B.hdr[i][0], B.hdr[i][1], r)[0] for i, r in enumerate(boxes))
    return full, sel


def crop_kernel_rate(cd, B, boxes):
    """k_crop_rows GB/s over (read + write) bytes of one region call, from the serialised per-kernel profile."""
    rd, rtotal = B.descs(boxes)
    rout = torch.empty(rtotal + 64, dtype=torch.uint8, device="cuda")
    cd.profile(True)
    cd.decode_region_raw(rd, rects(boxes), B.n, B.dev.data_ptr(), B.fsize, 1, B.foffs, B.fsizes, rout.data_ptr(), rtotal, 1)
    rep = cd.profile_report()
    cd.profile(False)
    nbytes = 2 * sum(w * h * B.hdr[i][2] for i, (_, _, w, h) in enumerate(boxes))
    ms = rep["k_crop_rows"][0]
    return {"crops": len(boxes), "bytes_read_plus_written": nbytes, "ms": round(ms, 4), "GBps": round(nbytes / ms / 1e6, 1)}


def timeline(cd, B, boxes, lv):
    """One full and one region decode of batch A with every launch bracketed by events (no host waits)."""
    fd, ftotal = B.descs()
    rd, rtotal = B.descs(boxes)
    fout = torch.empty(ftotal + 64, dtype=torch.uint8, device="cuda"); rout = torch.empty(rtotal + 64, dtype=torch.uint8, device="cuda")
    for what in ("full", "region"):
        for prof in (0, 3):
            cd.profile(prof)
            if prof:
                sys.stderr.write(f"TL level {lv}-{what}\n"); sys.stderr.flush()
            if what == "full":
                cd.decode_raw(fd, B.n, B.dev.data_ptr(), B.fsize, 1, B.foffs, B.fsizes, fout.data_ptr(), ftotal, 1)
            else:
                cd.decode_region_raw(rd, rects(boxes), B.n, B.dev.data_ptr(), B.fsize, 1, B.foffs, B.fsizes, rout.data_ptr(), rtotal, 1)
            sys.stderr.flush()
        cd.profile(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--timeline", action="store_true",
                    help="only the batch A calls under xpngb_profile(3): TL lines on stderr for tools/timeline_summary.py")
    a = ap.parse_args()
    if a.reps < 5:
        raise SystemExit("--reps must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("region_bench needs a CUDA device")
    res = {"tool": "tools/region_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3}
    cd = xpng_b200.Codec(0)

    # ---- A: the bench.py batch, one 224 x 224 crop per frame
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))
    rng = np.random.default_rng(2026)
    boxes = [(int(rng.integers(1920 - 224 + 1)), int(rng.integers(1080 - 224 + 1)), 224, 224) for _ in frames]
    A = {"frames": a.frames, "crop": [224, 224]}
    for lv in (1, 2):
        files = []
        for k in range(0, len(frames), 250):
            files += cd.encode(lv, frames[k: k + 250])
        B = Batch(files)
        if a.timeline:
            timeline(cd, B, boxes, lv)
            continue
        tf, tr = run_pair(cd, B, boxes, True, True, a.reps)
        nf, ns = tiles(B, boxes)
        A[f"L{lv}"] = {"full": tf, "region": tr, "tiles_full": nf, "tiles_region": ns, "tile_ratio": round(ns / nf, 4),
                       "time_ratio": round(tr["median_ms"] / tf["median_ms"], 4)}
        if lv == 1:
            res["C_crop_kernel_batch"] = crop_kernel_rate(cd, B, boxes)
        del B, files
        print(json.dumps({"A": {f"L{lv}": A[f"L{lv}"]}}), file=sys.stderr, flush=True)
    if a.timeline:
        return
    res["A_batch"] = A
    del frames

    # ---- B: single large images
    man = manifest()["synthetic"]
    Bres = {}
    for name in ("rgba_8192_s2", "rgb_4k_s1"):
        px = make_case("synthetic", name, man[name])
        H, W = px.shape[:2]
        for lv in (1, 2):
            f = cd.encode(lv, [px])[0]
            B = Batch([f])
            g = xpng_b200.region_tiles(W, H, (0, 0, W, H))
            cases = {"256": (W // 2 - 128, H // 2 - 128, 256, 256), "1024": (W // 2 - 512, H // 2 - 512, 1024, 1024)}
            grid = po.tile_grid(W, H)
            xs, ys = sorted(set(int(v) for v in grid[:, 0])), sorted(set(int(v) for v in grid[:, 1]))
            cases["2x2_tiles"] = (xs[1], ys[1], xs[3] - xs[1], ys[3] - ys[1])   # tile rows and columns 1..2: decoded in place
            cases["full"] = (0, 0, W, H)
            rec = {"tiles_full": g[0]}
            for cname, box in cases.items():
                r = {"rect": list(box), "tiles": xpng_b200.region_tiles(W, H, box)[0]}
                for where, dev in (("device", True), ("host", False)):
                    tf, tr = run_pair(cd, B, [box], dev, dev, a.reps)
                    r[where] = {"full": tf, "region": tr, "time_ratio": round(tr["median_ms"] / tf["median_ms"], 4)}
                rec[cname] = r
            if name == "rgba_8192_s2" and lv == 1:
                res["C_crop_kernel_8192_1024"] = crop_kernel_rate(cd, B, [cases["1024"]])
            Bres[f"{name}_L{lv}"] = rec
            print(json.dumps({"B": {f"{name}_L{lv}": rec}}), file=sys.stderr, flush=True)
            del B
    res["B_single"] = Bres
    cd.close()
    os.makedirs(os.path.join(ROOT, "profiles"), exist_ok=True)
    out = os.path.join(ROOT, "profiles", f"region_bench_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
