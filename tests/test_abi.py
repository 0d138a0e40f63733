"""CPU-side checks of the boundary: the C-ABI library loads and exports every symbol the headers
declare, host-only entry points behave like the reference (no GPU compute is called here)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT
import xpng_b200
from xpng_b200 import synth
from oracle import pyoracle as po


def declared_symbols():
    names = set()
    for h in ("xpng_b200.h", "xpng.h", "seven.h", "png7.h"):
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names |= set(re.findall(r"\b((?:xpngb?_|store_7|load_7|png_load|png_store|ppm_load|ppm_store|seven_main)\w*)\s*\(", src))
    return sorted(names)


def test_library_exports_every_declared_symbol():
    L = xpng_b200.lib()
    syms = declared_symbols()
    assert len(syms) >= 25
    for s in syms:
        assert hasattr(L, s), s


def test_no_cpu_fallback_without_device(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        xpng_b200.Codec(0)
    # the file API reports failure (returns 1) instead of silently using a CPU path
    assert xpng_b200.xpng_store(1, synth.rgb(8, 8, 1), str(tmp_path / "nogpu.xpng")) is True


def test_seven_container_roundtrip(tmp_path):
    for px in (synth.rgb(17, 31, 1), synth.rgba(9, 5, 2)):
        p = str(tmp_path / "a.7")
        assert xpng_b200.store_7(px, p) is False
        raw = open(p, "rb").read()
        ref = str(tmp_path / "b.7"); po.write_7(ref, px)
        assert raw == open(ref, "rb").read()
        assert np.array_equal(xpng_b200.load_7(p), px)
    # load_7 rejects short files, wrong mode byte, size mismatch (7/libseven.c:20-30)
    bad = tmp_path / "bad.7"
    bad.write_bytes(b"\0" * 10)
    with pytest.raises(RuntimeError):
        xpng_b200.load_7(str(bad))
    bad.write_bytes(raw[:8] + raw[8:-1])
    with pytest.raises(RuntimeError):
        xpng_b200.load_7(str(bad))
    bad.write_bytes(raw[:3] + b"\x01" + raw[4:])
    with pytest.raises(RuntimeError):
        xpng_b200.load_7(str(bad))


def test_peek_matches_oracle():
    L = xpng_b200.lib()
    from xpng_b200.codec import _Image
    for lv, px in ((1, synth.rgb(40, 50, 3)), (2, synth.rgba(33, 21, 4)), (7, synth.rgb(5, 6, 5))):
        f = po.encode(lv, px)
        d = _Image()
        b = np.frombuffer(f, dtype=np.uint8)
        assert L.xpngb_peek(b.ctypes.data, len(f), C.byref(d)) == 0
        assert (d.w, d.h, d.A, d.mode) == po.peek(f)
    assert L.xpngb_peek(np.zeros(8, np.uint8).ctypes.data, 8, C.byref(_Image())) == 1   # mode 0 is rejected (libxpng.c:972)


def test_cli_usage_and_stub(tmp_path):
    cli = os.path.join(ROOT, "xpng_b200", "bin", "xpng")
    r = subprocess.run([cli], capture_output=True, text=True)
    assert r.returncode == 1 and "encode: ./xpng -[127] example.7    example.xpng" in r.stdout
    r = subprocess.run([cli, "-3", "a.jpg", "b.xpng"], capture_output=True, text=True)
    assert r.returncode == 1 and "Not Implemented." in r.stdout      # libxpng.c:1004-1009
    r = subprocess.run([cli, "-1", str(tmp_path / "missing.7"), str(tmp_path / "o.xpng")], capture_output=True, text=True)
    assert r.returncode == 1


def test_encode_bound():
    from xpng_b200.codec import Codec
    d, total = Codec.layout([(10, 20, 3), (7, 9, 4)])
    assert d[1].offset == 608 and total == 608 + 256
    assert xpng_b200.lib().xpngb_encode_bound(d, 2) == 608 + 272
