#!/usr/bin/env python
"""Encode-side A/B of builds of the library on bench.py's batch (sintel-like 1920x1080 RGB frames, seeds 1000.., pixels
and files in HBM), one process, the builds alternated run by run:

    python tools/front2_ab.py [--lib PATH ...] [--runs 3] [--frames 1000] [--out profiles/NAME.json]

Per build and run:
  kernels  every encode kernel summed over one level-1 and one level-2 call, CUDA events per launch with the launches
           serialised (xpngb_profile, as bench.py's breakdown.kernels_ms_rank0); k_front2<1> / k_front2<2> are the RGB front end;
  alone    the level-1 and the level-2 encode call one at a time (median of three; the call returns with its work done);
  both     the two calls at once, one codec context and host thread each, as a bench.py step starts (median of three).
The encoded files of every build are hashed: builds that differ in speed only give the same `files_sha`.  The GPU's name,
power limit and SM clock are read in the same run.  Without --lib the build in xpng_b200/ is measured."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import xpng_b200  # noqa: E402
from xpng_b200 import codec, synth, Codec  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), (v.strip() for v in out.strip().split(","))))


def use_lib(path):
    """Point the ctypes mirror at another build; contexts of the previous one must be closed first."""
    os.environ["XPNGB_LIB"] = os.path.abspath(path)
    codec._lib = None
    return xpng_b200.lib()


def measure(lib_path, d_px, shapes, total, d_out, cap, want_sha):
    lib = use_lib(lib_path)
    n = len(shapes)
    cds = {lv: Codec(0) for lv in (1, 2)}

    def enc(lv):
        d, _ = Codec.layout(shapes)
        t0 = time.perf_counter()
        offs, sizes = cds[lv].encode_raw(lv, d, n, d_px.data_ptr(), total, 1, d_out[lv].data_ptr(), cap, 1)
        return (time.perf_counter() - t0) * 1e3, offs, sizes

    rec = {"lib": lib_path}
    for lv in (1, 2):
        enc(lv)                                                  # warm-up: buffers, modules
    rec["alone_ms"] = {f"enc{lv}": round(statistics.median(enc(lv)[0] for _ in range(3)), 3) for lv in (1, 2)}
    both = {"enc1": [], "enc2": [], "pair": []}
    for _ in range(3):
        res = {}
        ths = [threading.Thread(target=lambda lv=lv: res.__setitem__(lv, enc(lv)[0])) for lv in (2, 1)]
        t0 = time.perf_counter()
        for t in ths: t.start()
        for t in ths: t.join()
        both["pair"].append((time.perf_counter() - t0) * 1e3)
        both["enc1"].append(res[1]); both["enc2"].append(res[2])
    rec["both_ms"] = {k: round(statistics.median(v), 3) for k, v in both.items()}
    kern = {}
    for lv in (1, 2):
        cds[lv].profile(True)
        _, offs, sizes = enc(lv)
        for k, (ms, cnt) in cds[lv].profile_report().items():
            kern[f"L{lv}.enc.{k}"] = round(ms, 3)
        cds[lv].profile(False)
        if want_sha:
            h = hashlib.sha256(np.array(list(sizes), np.uint64).tobytes())
            used = int(max(o + s for o, s in zip(offs, sizes)))
            h.update(d_out[lv][:used].cpu().numpy().tobytes())
            rec[f"files_sha_L{lv}"] = h.hexdigest()[:16]
    rec["kernels_ms"] = dict(sorted(kern.items(), key=lambda kv: -kv[1]))
    for c in cds.values():
        c.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", help="library build to measure (repeat for an A/B; default: xpng_b200/libxpng_b200.so)")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--out", help="write the JSON record here as well")
    args = ap.parse_args()
    libs = args.lib or [codec.lib_path()]
    info = {"before": gpu_info()}
    frames = synth.sintel_batch(range(1000, 1000 + args.frames))
    shapes = [f.shape for f in frames]
    descs, total = Codec.layout(shapes)
    buf = np.zeros(total + 64, np.uint8)
    for d, f in zip(descs, frames):
        buf[d.offset:d.offset + f.size] = f.reshape(-1)
    del frames
    use_lib(libs[0])
    cap = int(xpng_b200.lib().xpngb_encode_bound(descs, args.frames))
    d_px = torch.from_numpy(buf).cuda()
    d_out = {lv: torch.zeros(cap + 64, dtype=torch.uint8, device="cuda") for lv in (1, 2)}
    runs = []
    for r in range(args.runs):
        for lp in (libs if r % 2 == 0 else libs[::-1]):
            rec = measure(lp, d_px, shapes, total, d_out, cap, want_sha=r == 0)
            rec["run"] = r
            runs.append(rec)
            print(json.dumps(rec), flush=True)
    info["after"] = gpu_info()
    summary = {}
    for lp in libs:
        rs = [x for x in runs if x["lib"] == lp]
        row = {}
        for key in ("alone_ms", "both_ms"):
            for k in rs[0][key]:
                v = [x[key][k] for x in rs]
                row[f"{key[:-3]}.{k}"] = {"median": round(statistics.median(v), 3), "min": min(v), "max": max(v)}
        for k in ("L1.enc.k_front2<1>", "L2.enc.k_front2<2>"):
            v = [x["kernels_ms"].get(k, 0.0) for x in rs]
            row[k] = {"median": round(statistics.median(v), 3), "min": min(v), "max": max(v)}
        row["files_sha"] = [rs[0].get("files_sha_L1"), rs[0].get("files_sha_L2")]
        summary[lp] = row
    out = {"what": "encode A/B on sintel-like 1080p frames in HBM (tools/front2_ab.py)", "frames": args.frames, "runs_per_lib": args.runs,
           "gpu": info, "summary": summary, "runs": runs}
    print(json.dumps({"summary": summary, "gpu": info}, indent=1), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(out, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
