#!/usr/bin/env python
"""Auto-augmented decode on the GPU; one JSON line to profiles/augment_decode_<tag>.json.  Files and outputs in device memory.

The workload is the colour bench's batch with a supervised policy instead of the colour step: sintel-like 1080p frames at
levels 1 and 2, each with a seeded RandomResizedCrop box resized (bilinear) to 224 x 224 and a horizontal flip with p 0.5, then
TrivialAugmentWide(bilinear) or RandAugment(2, 9) replayed from torch's RNG, written as an ImageNet-normalised float32
(N, 3, 224, 224) tensor.  The arms, called in turn:
  floor    tensor decode of the same boxes and flips without the policy (xpngb_decode_resampled)
  augment  the whole view in one xpngb_decode_augment call
  host_pil uint8 decode (xpngb_decode_resized), copy to the host, torchvision's policy on each PIL image, PILToTensor, back to
           the device, then ToDtype + Normalize there
A sample of the augment arm is compared with Pillow (torchvision's _apply_op on the PIL crop) first.  Each timing is 3 warm-up
calls, then --reps calls per arm, each ending in a device synchronise; the median is reported.  Per-kernel times of one
augment call come from xpngb_profile.
Usage: python tools/augment_decode_bench.py [--frames 1000] [--reps 7] [--tag b200] [--out FILE]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from region_bench import Batch, gpu_info  # noqa: E402  (also puts the repository and tests/ on sys.path)
import torch  # noqa: E402
import xpng_b200  # noqa: E402
from xpng_b200 import synth  # noqa: E402
from xpng_b200.codec import (_Image, augment_array, augment_params, op_codes, rand_augment_ops, rects, sizes,  # noqa: E402
                             tensor_format, trivial_augment_wide_ops)
from oracle import pyoracle as po  # noqa: E402
from test_resized_decode import rrc_boxes  # noqa: E402
from test_resampled_decode import resize_pil  # noqa: E402
from test_tensor_decode import bits, to_tensor_ref  # noqa: E402
from resampled_decode_bench import alternate  # noqa: E402

OUT = (224, 224)
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def programs(policy, n, seed):
    """Flip, _apply_op steps and their program per frame, drawn as RandomHorizontalFlip and the policy's forward do."""
    replay = trivial_augment_wide_ops if type(policy).__name__ == "TrivialAugmentWide" else rand_augment_ops
    torch.manual_seed(seed)
    ops, steps = [], []
    for _ in range(n):
        ops.append("mh" if torch.rand(1) < 0.5 else "tl")
        steps.append(replay(policy, OUT))
    return ops, steps, [augment_params(st, OUT, policy.interpolation, policy.fill) for st in steps]


def run_level(cd, files, boxes, policy, seed, reps):
    from PIL import Image
    from torchvision.transforms import functional as F
    n = len(files)
    ops, steps, augs = programs(policy, n, seed)
    B = Batch(files)
    fptr = B.dev.data_ptr()
    ra, sa, oa, aa = rects(boxes), sizes([OUT] * n), op_codes(ops), augment_array(augs, n)
    fmt = tensor_format("float32", "chw", "div", MEAN, STD, drop_alpha=True)
    per = 3 * OUT[0] * OUT[1]
    td = (_Image * n)()
    ud = (_Image * n)()
    for i in range(n):
        td[i].offset, ud[i].offset = i * per * 4, i * per
    t_floor = torch.empty((n, 3, *OUT[::-1]), dtype=torch.float32, device="cuda")
    t_aug = torch.empty_like(t_floor)
    u8 = torch.empty((n, OUT[1], OUT[0], 3), dtype=torch.uint8, device="cuda")
    mean = torch.tensor(MEAN, device="cuda").view(3, 1, 1)
    std = torch.tensor(STD, device="cuda").view(3, 1, 1)

    floor = lambda: cd.decode_resampled_raw(fmt, td, None, oa, ra, sa, None, n, fptr, B.fsize, 1, B.foffs, B.fsizes, t_floor.data_ptr(),
                                            n * per * 4, 1)
    augment = lambda: cd.decode_augment_raw(fmt, td, None, oa, ra, sa, None, None, None, aa, n, fptr, B.fsize, 1, B.foffs, B.fsizes,
                                            t_aug.data_ptr(), n * per * 4, 1)

    def host_pil():
        cd.decode_resized_raw(ud, oa, ra, sa, n, fptr, B.fsize, 1, B.foffs, B.fsizes, u8.data_ptr(), n * per, 1)
        host = u8.cpu().numpy()
        out = torch.stack([F.pil_to_tensor(policy(Image.fromarray(host[i]))) for i in range(n)])
        return out.cuda().float().mul_(1 / 255).sub_(mean).div_(std)

    # correctness of the augment arm on a sample: against the restatement
    from torchvision.transforms.autoaugment import _apply_op
    from test_augment_decode import augment_ref
    augment(); torch.cuda.synchronize()
    for i in range(0, n, max(1, n // 40)):
        x, y, w, h = boxes[i]
        px = po.orient(ops[i], resize_pil(po.decode(files[i])[y: y + h, x: x + w], *OUT, 2))
        want = augment_ref(px, augs[i])
        if not np.array_equal(bits(t_aug[i]), to_tensor_ref(want, "float32", "chw", "div", MEAN, STD)):
            raise SystemExit(f"entry {i}: augment decode differs from the restatement")
    # and against Pillow itself: torchvision's _apply_op on the PIL crop, with the same draws
    for i in range(0, n, max(1, n // 40)):
        x, y, w, h = boxes[i]
        img = Image.fromarray(po.orient(ops[i], resize_pil(po.decode(files[i])[y: y + h, x: x + w], *OUT, 2)))
        for name, m in steps[i]:
            img = _apply_op(img, name, m, interpolation=policy.interpolation, fill=policy.fill)
        if not np.array_equal(bits(t_aug[i]), to_tensor_ref(np.asarray(img), "float32", "chw", "div", MEAN, STD)):
            raise SystemExit(f"entry {i}: augment decode differs from torchvision's PIL path")
    cd.profile(True)
    augment()
    prof = {k: v for k, v in cd.profile_report().items() if k.startswith(("k_aug", "k_color")) or k == "k_to_tensor"}
    cd.profile(False)
    r = alternate({"floor_tensor_no_policy": floor, "augment_decode": augment, "host_pil_policy": host_pil}, reps)
    r["profiled_one_call_ms"] = {k: round(v[0], 3) for k, v in prof.items()}
    r["augment_steps"] = sum(a.nsteps for a in augs)
    del B
    return r


def main():
    import torchvision.transforms as T
    from torchvision.transforms import InterpolationMode as IM
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", help="output file (default profiles/augment_decode_<tag>.json)")
    a = ap.parse_args()
    if a.reps < 5:
        raise SystemExit("--reps must be at least 5")
    if not torch.cuda.is_available():
        raise SystemExit("augment_decode_bench needs a CUDA device")
    res = {"tool": "tools/augment_decode_bench.py", **gpu_info(), "reps": a.reps, "warmup": 3, "frames": a.frames, "size": list(OUT)}
    cd = xpng_b200.Codec(0)
    frames = synth.sintel_batch(range(1000, 1000 + a.frames))
    boxes = rrc_boxes(np.random.default_rng(2029), len(frames))
    policies = {"trivial_augment_wide_bilinear": T.TrivialAugmentWide(interpolation=IM.BILINEAR),
                "rand_augment_2_9": T.RandAugment(2, 9)}
    for lv in (1, 2):
        files = []
        for k in range(0, len(frames), 250):
            files += cd.encode(lv, frames[k: k + 250])
        for pname, pol in policies.items():
            key = f"{pname}_224_f32_L{lv}"
            res[key] = run_level(cd, files, boxes, pol, 2030 + lv, a.reps)
            print(key, json.dumps(res[key]), file=sys.stderr, flush=True)
    cd.close()
    out = a.out or os.path.join(ROOT, "profiles", f"augment_decode_{a.tag}.json")
    line = json.dumps(res)
    with open(out, "w") as fh:
        fh.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
