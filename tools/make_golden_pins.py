#!/usr/bin/env python
"""Writes tests/golden/reference_pins.json: what the reference comparisons of the suite compare against, so that a checkout
without the reference build still runs them:
  oracle_vs_reference  tests/test_oracle_pin.py::test_oracle_matches_reference_binary (size and sha256 of each file, sha256
                       of its decoded pixels, per seed and level)
  orient               tests/test_orient.py::test_restatement_matches_reference_tool (shape and sha256 of each output)
  file_api_cli         tests/test_gpu_parity.py::test_file_api_and_cli_against_reference (sha256 of each file)

With the reference built into oracle/_ref (oracle/Makefile) the values come from the reference binary and tool themselves.
Without it they come from the oracle (oracle/xpng_oracle.c) and the numpy restatement (pyoracle.orient), which those tests
compared equal with the reference build on these inputs; "source" in the file records which was used.
Usage: python tools/make_golden_pins.py [--source-note TEXT]"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from oracle import pyoracle as po  # noqa: E402
import test_gpu_parity  # noqa: E402
import test_oracle_pin  # noqa: E402
import test_orient  # noqa: E402


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


def main():
    ref = po.ref_available() and os.path.exists(po.REF_TOOL)
    encode = po.ref_encode if ref else po.encode
    decode = po.ref_decode if ref else po.decode
    orient = po.ref_orient if ref else po.orient
    note = sys.argv[sys.argv.index("--source-note") + 1] if "--source-note" in sys.argv else ""
    out = {"source": ("the reference build (oracle/_ref)" if ref else "the oracle and the numpy restatement") + (": " + note if note else ""),
           "oracle_vs_reference": {}, "orient": {}, "file_api_cli": {}}
    for seed in range(6):
        px = test_oracle_pin.random_case(seed)
        e = out["oracle_vs_reference"][str(seed)] = {"shape": list(px.shape), "decoded_shape": list(po.normalize(px).shape)}
        for lv in (1, 2, 7):
            f = encode(lv, px)
            e[str(lv)] = {"size": len(f), "sha256": sha(f), "decoded_sha256": sha(decode(f).tobytes())}
    for op in po.TOOL_OPS:
        out["orient"][op] = {}
        for shape in test_orient.SHAPES:
            o = orient(op, test_orient._px(shape))
            out["orient"][op]["x".join(map(str, shape))] = [list(o.shape), sha(o.tobytes())]
    for key, (gen, h, w, seed) in test_gpu_parity.CLI_CASES.items():
        px = gen(h, w, seed)
        out["file_api_cli"][key] = {str(lv): sha(encode(lv, px)) for lv in (1, 2, 7)}
    with open(os.path.join(ROOT, "tests", "golden", "reference_pins.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
