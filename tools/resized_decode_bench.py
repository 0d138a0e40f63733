#!/usr/bin/env python
"""Resized decode against what callers do without it, on the GPU; one JSON line to profiles/resized_decode_<tag>.json.

  A  the bench.py workload (1000 sintel-like 1080p frames, seeds 1000..), levels 1 and 2, one seeded RandomResizedCrop-style
     box per frame (area share U(0.08, 1), aspect log-uniform in [3/4, 4/3]) resized to 224 x 224, MH on a seeded half
     (TL, a copy, on the rest).  Paths, with files and pixels in device memory and again in pinned host memory:
       crops_only        xpngb_decode_oriented of the boxes (the crops, not resized: the lower bound)
       decode_resized    xpngb_decode_resized
       today             device: decode_oriented + one torch.nn.functional.interpolate(bilinear, antialias=True) per crop
                         (a cost reference only: its float output is not Pillow's); host: decode_oriented + PIL
                         Image.resize(BILINEAR) of each crop on the host cores, timed on the first --pil-sample crops and
                         scaled to the batch (labelled as such).
  B  rgb_4k_s1 and rgba_8192_s2, whole image -> 224 x 224: xpngb_decode against xpngb_decode_resized, device and host.
  K  the resize kernels' own time (xpngb_profile: launches serialised, a run of its own) for A at level 1 in device
     memory, and the bytes the passes must read and write (from the shapes) over that time.

Before anything is timed, a sample of every path's outputs is compared with the oracle (tests/test_resized_decode.py:
resize_bilinear, Pillow's bilinear resize restated).  A timing is 3 warm-up calls and then `--reps` calls, each ending in a
device synchronise; median and minimum are reported, with xpngb_last_kernel_ms of the last call.
Usage: python tools/resized_decode_bench.py [--frames 1000] [--reps 7] [--pil-sample 100] [--tag b200]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from region_bench import Batch, gpu_info, timed  # noqa: E402  (also puts the repository and tests/ on sys.path)
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
from PIL import Image  # noqa: E402
import xpng_b200  # noqa: E402
from xpng_b200 import synth  # noqa: E402
from xpng_b200.codec import _Image, op_codes, rects, sizes  # noqa: E402
from conftest import make_case, manifest  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from test_resized_decode import resize_bilinear, rrc_boxes  # noqa: E402

OUT = (224, 224)


def out_descs(B, whs):
    """Output layout: entry i is whs[i] = (w, h) pixels."""
    arr, off = (_Image * B.n)(), 0
    for i, (w, h, c) in enumerate(B.hdr):
        arr[i].offset = off
        off += (whs[i][0] * whs[i][1] * c + 15) & ~15
    return arr, off


def buf(nbytes, dev):
    t = torch.zeros(nbytes + 64, dtype=torch.uint8, device="cuda" if dev else "cpu")
    return t if dev else t.pin_memory()


def entry(t, d, w, h, c):
    return t[d.offset: d.offset + w * h * c].reshape(h, w, c)


def check_sample(files, boxes, ops, got, k):
    """Entries 0, k, 2k, ... of `got` (numpy (h, w, c) of the 224 x 224 outputs) against the oracle."""
    for i in range(0, len(files), k):
        full = po.decode(files[i])
        x, y, w, h = boxes[i] if boxes is not None else (0, 0, full.shape[1], full.shape[0])
        want = po.orient(ops[i] if ops else "tl", resize_bilinear(full[y: y + h, x: x + w], *OUT))
        if not np.array_equal(got(i), want):
            raise SystemExit(f"parity: entry {i} differs from the oracle")


def batch_paths(cd, B, files, boxes, ops, dev, reps, pil_sample):
    fptr = B.dev.data_ptr() if dev else B.host.ctypes.data
    n = B.n
    ra, oa, sa = rects(boxes), op_codes(ops), sizes([OUT] * n)
    dc, tc = out_descs(B, [b[2:] for b in boxes])
    dr, tr = out_descs(B, [OUT] * n)
    crops, resized = buf(tc, dev), buf(tr, dev)

    def crops_only():
        cd.decode_oriented_raw(dc, oa, ra, n, fptr, B.fsize, int(dev), B.foffs, B.fsizes, crops.data_ptr(), tc, int(dev))

    def dec_resized():
        cd.decode_resized_raw(dr, oa, ra, sa, n, fptr, B.fsize, int(dev), B.foffs, B.fsizes, resized.data_ptr(), tr, int(dev))

    dec_resized(); torch.cuda.synchronize()
    host = resized.cpu().numpy()
    check_sample(files, boxes, ops, lambda i: entry(host, dr[i], *OUT, B.hdr[i][2]), 50)
    out = {"crops_only": timed(crops_only, reps)}
    out["crops_only"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
    out["decode_resized"] = timed(dec_resized, reps)
    out["decode_resized"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
    out["crop_bytes"], out["resized_bytes"] = tc, tr
    if dev:
        views = [entry(crops, dc[i], boxes[i][2], boxes[i][3], B.hdr[i][2]).permute(2, 0, 1)[None] for i in range(n)]

        def today():
            crops_only()
            return [F.interpolate(v.float(), size=OUT[::-1], mode="bilinear", antialias=True, align_corners=False) for v in views]

        out["today_decode_oriented_plus_interpolate_per_crop"] = timed(today, reps)
        out["today_decode_oriented_plus_interpolate_per_crop"]["note"] = "one interpolate launch per crop; float output, not Pillow's"
    else:
        crops_only(); torch.cuda.synchronize()
        hc = crops.numpy()
        m = min(pil_sample, n)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            for i in range(m):
                Image.fromarray(entry(hc, dc[i], boxes[i][2], boxes[i][3], B.hdr[i][2])).resize(OUT, Image.BILINEAR)
            ts.append((time.perf_counter() - t0) * 1e3)
        pil_ms = float(np.median(ts)) * n / m
        out["today_pil_resize_on_host_scaled_ms"] = {"ms": round(pil_ms, 3), "sampled_crops": m, "threads": 1,
                                                     "note": f"PIL resize of {m} crops, one thread, scaled by {n}/{m}"}
        out["today_decode_oriented_plus_pil_ms"] = round(out["crops_only"]["median_ms"] + pil_ms, 3)
    return out


def resize_kernel_rate(cd, B, boxes, ops):
    """K: per-kernel time of the resize launches (profiled run) and the bytes the two passes must move."""
    n = B.n
    dr, tr = out_descs(B, [OUT] * n)
    out_t = buf(tr, True)
    ra, oa, sa = rects(boxes), op_codes(ops), sizes([OUT] * n)
    cd.profile(True)
    calls = 3
    for _ in range(calls):
        cd.decode_resized_raw(dr, oa, ra, sa, n, B.dev.data_ptr(), B.fsize, 1, B.foffs, B.fsizes, out_t.data_ptr(), tr, 1)
    rep = cd.profile_report()
    cd.profile(False)
    hb = vb = 0
    for (x, y, w, h), (_, _, c) in zip(boxes, B.hdr):
        tmp = h * OUT[0] * c
        hb += w * h * c + tmp                      # horizontal pass: the crop in, in_h rows of 224 pixels out
        vb += tmp + OUT[0] * OUT[1] * c            # vertical pass: those rows in, the output out
    res = {}
    for name, nbytes in (("k_resize_coeffs", 0), ("k_resize_h", hb), ("k_resize_v", vb)):
        ms, cnt = rep.get(name, (0.0, 0))
        per = ms / calls                           # one launch per chunk: the call's launches together
        res[name] = {"ms_per_call": round(per, 4), "launches_per_call": cnt // calls, "bytes": nbytes,
                     "GB_per_s": round(nbytes / per / 1e6, 1) if nbytes and per else None}
    res["other_kernels_ms_per_call"] = round(sum(v[0] for k, v in rep.items() if not k.startswith("k_resize")) / calls, 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--pil-sample", type=int, default=100)
    ap.add_argument("--tag", default="b200")
    a = ap.parse_args()
    if a.reps < 5:
        raise SystemExit("--reps must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("resized_decode_bench needs a CUDA device")
    res = {"tool": "tools/resized_decode_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3, "size": list(OUT)}
    cd = xpng_b200.Codec(0)

    # ---- A and K: the bench.py batch
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))
    rng = np.random.default_rng(2028)
    boxes = rrc_boxes(rng, len(frames))
    ops = [("mh", "tl")[int(rng.integers(2))] for _ in frames]
    files = {}
    for lv in (1, 2):
        files[lv] = []
        for k in range(0, len(frames), 250):
            files[lv] += cd.encode(lv, frames[k: k + 250])
    del frames
    A = {"frames": a.frames, "boxes": "RandomResizedCrop-style, seeded", "mean_box_pixels": round(float(np.mean([b[2] * b[3] for b in boxes]))),
         "mh_entries": ops.count("mh")}
    for lv in (1, 2):
        B = Batch(files[lv])
        for where, dev in (("device", True), ("host", False)):
            A[f"L{lv}_{where}"] = batch_paths(cd, B, files[lv], boxes, ops, dev, a.reps, a.pil_sample)
            print(json.dumps({"A": {f"L{lv}_{where}": A[f"L{lv}_{where}"]}}), file=sys.stderr, flush=True)
        if lv == 1:
            res["K_resize_kernels_L1_device"] = resize_kernel_rate(cd, B, boxes, ops)
            print(json.dumps({"K": res["K_resize_kernels_L1_device"]}), file=sys.stderr, flush=True)
        del B
    res["A_batch_rrc_224"] = A
    del files

    # ---- B: single large images, whole -> 224 x 224
    man = manifest()["synthetic"]
    Bres = {}
    for name in ("rgb_4k_s1", "rgba_8192_s2"):
        px = make_case("synthetic", name, man[name])
        for lv in (1, 2):
            f = cd.encode(lv, [px])
            B = Batch(f)
            for where, dev in (("device", True), ("host", False)):
                fptr = B.dev.data_ptr() if dev else B.host.ctypes.data
                df, tf = B.descs()
                dr, tr = out_descs(B, [OUT])
                full, small = buf(tf, dev), buf(tr, dev)
                sa = sizes([OUT])

                def dec():
                    cd.decode_raw(df, 1, fptr, B.fsize, int(dev), B.foffs, B.fsizes, full.data_ptr(), tf, int(dev))

                def res_():
                    cd.decode_resized_raw(dr, None, None, sa, 1, fptr, B.fsize, int(dev), B.foffs, B.fsizes, small.data_ptr(), tr, int(dev))

                res_(); torch.cuda.synchronize()
                h = small.cpu().numpy()
                check_sample(f, None, None, lambda i: entry(h, dr[i], *OUT, B.hdr[i][2]), 1)
                r = {"decode": timed(dec, a.reps)}
                r["decode"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
                r["decode_resized"] = timed(res_, a.reps)
                r["decode_resized"]["kernel_ms"] = round(cd.last_kernel_ms, 3)
                Bres[f"{name}_L{lv}_{where}"] = r
                print(json.dumps({"B": {f"{name}_L{lv}_{where}": r}}), file=sys.stderr, flush=True)
            del B
    res["B_thumbnail_224"] = Bres
    cd.close()
    out = os.path.join(ROOT, "profiles", f"resized_decode_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
