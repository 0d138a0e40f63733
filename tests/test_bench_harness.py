"""Host-side pieces of bench.py that can be checked without a GPU: the file-API harness (against oracle/libxo_file.so, the
xpng_store_T / xpng_load_T entry points of the drop-in over the CPU oracle, and against the reference library when it is built
into oracle/_ref), the --dump-outputs writer and the NUMA binding helper."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from oracle import pyoracle as po  # noqa: E402
from xpng_b200 import synth  # noqa: E402

FILE_LIB = os.path.join(ROOT, "oracle", "libxo_file.so")
REF = os.path.join(ROOT, "oracle", "_ref", "libxpng_ref.so")


def _file_lib():
    if not os.path.exists(FILE_LIB):
        po.build()
    return C.CDLL(FILE_LIB)


@pytest.mark.parametrize("callers", [1, 3])
def test_file_api_steps_one_and_many_callers(callers):
    """Every frame is stored and loaded at levels 1 and 2, from one caller or several; no file is left behind.
    Run against the oracle's file library, and against the reference library that --impl reference times when it is built."""
    frames = [synth.sintel_like(1000 + k, 270, 480) for k in range(3)]
    for L in [_file_lib()] + ([C.CDLL(REF)] if os.path.exists(REF) else []):
        per_step, calls = bench.file_api_steps(L, frames, 1, 1, f"t{callers}", callers=callers)
        assert per_step > 0 and set(calls) == {"enc1", "dec1", "enc2", "dec2"} and all(v > 0 for v in calls.values())
        assert not [f for f in os.listdir(bench._tmpdir()) if f.startswith(f"_xpng_t{callers}_{os.getpid()}_")]


def test_oracle_file_api_writes_and_reads_oracle_files(tmp_path):
    """The harness's CPU library: xpng_store_T writes the oracle's file, xpng_load_T returns the normalised pixels."""
    L = _file_lib()
    L.xpng_store_T.argtypes = [C.c_uint64, C.c_uint64, C.POINTER(bench._Xpng), C.c_char_p]
    L.xpng_load_T.argtypes = [C.c_uint64, C.c_char_p, C.POINTER(bench._Xpng)]
    L.xpng_store_T.restype = L.xpng_load_T.restype = C.c_bool
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    path = str(tmp_path / "a.xpng").encode()
    for lv, px in ((1, synth.rgb(70, 90, 3)), (2, synth.rgba(40, 50, 4)), (7, synth.rgb(5, 6, 5))):
        assert not L.xpng_store_T(0, lv, C.byref(bench._Xpng(px.ctypes.data, px.shape[1], px.shape[0], px.size, px.shape[2] == 4)), path)
        assert open(path, "rb").read() == po.encode(lv, px)
        out = bench._Xpng()
        assert not L.xpng_load_T(0, path, C.byref(out))
        got = np.ctypeslib.as_array(C.cast(out.p, C.POINTER(C.c_uint8)), shape=(out.s,)).reshape(out.h, out.w, 3 + out.A).copy()
        libc.free(out.p)
        assert np.array_equal(got, po.normalize(px))
    assert L.xpng_store_T(0, 3, C.byref(bench._Xpng(px.ctypes.data, px.shape[1], px.shape[0], px.size, False)), path)   # mode 3
    assert L.xpng_load_T(0, str(tmp_path / "missing.xpng").encode(), C.byref(bench._Xpng()))


@pytest.mark.parametrize("file_sample", [None, 100])
def test_dump_outputs_writes_the_files_in_frame_order_and_a_fixed_sample(tmp_path, monkeypatch, file_sample):
    """Every file byte in frame order (None), or a fixed sample of 100 positions of that concatenation; a fixed sample of the
    decoded arena; the same arrays on every run."""
    import torch
    files = [po.encode(lv, synth.rgb(30 + lv, 40, lv)) for lv in (1, 2)]
    arena = np.zeros(256 + sum(len(f) for f in files), np.uint8)
    offs = [len(files[1]) + 48, 16]                           # the files lie in the arena out of frame order, with gaps
    for o, f in zip(offs, files):
        arena[o:o + len(f)] = np.frombuffer(f, np.uint8)
    back = np.random.default_rng(3).integers(0, 256, 1000, dtype=np.uint8)
    t = {lv: torch.from_numpy(arena) for lv in bench.LEVELS}
    b = {lv: torch.from_numpy(back) for lv in bench.LEVELS}
    monkeypatch.setattr(bench, "DUMP_PIXEL_BYTES", 64)
    if file_sample:
        monkeypatch.setattr(bench, "DUMP_FILE_BYTES", file_sample)
    concat = np.frombuffer(b"".join(files), np.uint8)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), t, b, {lv: offs for lv in bench.LEVELS}, {lv: [len(f) for f in files] for lv in bench.LEVELS}, 1000)
    for lv in bench.LEVELS:
        got = {k: np.load(str(tmp_path / "a" / f"L{lv}_{k}.npy")) for k in ("sizes", "offsets", "file_bytes", "decoded_pixels")}
        assert got["sizes"].dtype == np.float64 and got["sizes"].tolist() == [len(f) for f in files] and got["offsets"].tolist() == offs
        want = concat if not file_sample else concat[bench._sample_positions(len(concat), file_sample, lv)]
        assert len(want) == (file_sample or len(concat))
        assert got["file_bytes"].dtype == np.float32 and np.array_equal(got["file_bytes"], want.astype(np.float32))
        px = got["decoded_pixels"]
        assert px.dtype == np.float32 and np.array_equal(px, back[bench._sample_positions(1000, 64, 100 + lv)].astype(np.float32))
        for k, v in got.items():
            assert np.array_equal(v, np.load(str(tmp_path / "b" / f"L{lv}_{k}.npy"))), k      # the same sample every run


def test_bind_near_gpu_never_raises_and_keeps_the_affinity_without_a_gpu():
    before = os.sched_getaffinity(0)
    rec, orig = bench.bind_near_gpu(0)
    try:
        assert orig == before and isinstance(rec, dict) and "numa_node" in rec
        assert os.sched_getaffinity(0) <= before
    finally:
        os.sched_setaffinity(0, before)
