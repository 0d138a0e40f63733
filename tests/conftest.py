import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")
CORPUS = os.path.join(GOLD, "corpus")             # the reference's images/*.png (test inputs of config 0), committed


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "slow: full BASELINE sizes on the CPU oracle")


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def load_png(path):
    from PIL import Image
    im = Image.open(path)
    im = im.convert("RGBA" if ("A" in im.getbands() or "transparency" in im.info) else "RGB")
    return np.ascontiguousarray(np.asarray(im, dtype=np.uint8))


def manifest():
    with open(os.path.join(GOLD, "manifest.json")) as f:
        return json.load(f)


def make_case(group, name, entry):
    """Rebuild the input pixels of a manifest entry."""
    from xpng_b200 import synth
    if group == "crops":
        return load_png(os.path.join(GOLD, "crops", name))
    if group == "corpus":
        p = os.path.join(CORPUS, name)
        assert os.path.exists(p), f"{p} is missing: the config-0 corpus is a committed fixture (tools/make_golden.py)"
        return load_png(p)
    fn, args = entry["gen"]
    if fn == "full":
        return np.full(tuple(args[0]), args[1], np.uint8)
    if fn == "opaque":
        h, w, s = args
        return np.concatenate([synth.rgb(h, w, s), np.full((h, w, 1), 255, np.uint8)], axis=2)
    if fn == "dirty":
        d = synth.rgba(*args); d[d[..., 3] == 0] = [9, 8, 7, 0]; return d
    if fn == "halfflat":
        d = synth.rgb(*args); d[:, :450] = [10, 200, 30]; return d
    return getattr(synth, fn)(*args)


BIG = {"rgb_4k_s1", "gray_4096_s3000", "rgba_8192_s2"}


def reference_pins():
    """What the reference comparisons of the suite compare against (tools/make_golden_pins.py)."""
    with open(os.path.join(GOLD, "reference_pins.json")) as f:
        return json.load(f)


def all_cases(groups=("synthetic", "special", "crops"), big=False):
    man = manifest()
    out = []
    for g in groups:
        for name, e in sorted(man[g].items()):
            if name in BIG and not big:
                continue
            out.append((g, name, e))
    return out
