"""ctypes front end of the CPU oracle (oracle/liboracle.so) and, when built, of the unmodified
reference (oracle/_ref/libxpng_ref.so, oracle/_ref/xpng).

TEST INFRASTRUCTURE ONLY — imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; never by the product package xpng_b200.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(HERE, "liboracle.so")
_REF_DIR = os.path.join(HERE, "_ref")
_REF_LIB = os.path.join(_REF_DIR, "libxpng_ref.so")
REF_CLI = os.path.join(_REF_DIR, "xpng")


def build():
    subprocess.run(["make", "-s", "-C", HERE], check=True)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            build()
        L = C.CDLL(_LIB)
        u8p, u64, u32p = C.POINTER(C.c_uint8), C.c_uint64, C.POINTER(C.c_uint32)
        L.xo_tile_grid.restype = u64
        L.xo_tile_grid.argtypes = [u64, u64, C.c_int, C.c_void_p, u64]
        L.xo_normalize.restype = C.c_int
        L.xo_normalize.argtypes = [C.c_void_p, u64, u64, C.c_int, C.c_void_p, C.POINTER(u64)]
        L.xo_select_predictor.restype = C.c_uint
        L.xo_select_predictor.argtypes = [C.c_void_p, u64, u64, u64, C.c_int]
        L.xo_m1_front.restype = u64
        L.xo_m1_front.argtypes = [C.c_void_p, u64, u64, u64, C.c_int, C.c_uint, C.c_void_p, u32p, u32p, C.c_void_p]
        L.xo_block_v2_encode.restype = u64
        L.xo_block_v2_encode.argtypes = [u32p, C.c_uint, C.c_void_p, u64, C.c_void_p, C.c_int]
        L.xo_block_v2_decode.restype = u64
        L.xo_block_v2_decode.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(u64)]
        L.xo_encode_tile_m1.restype = u64
        L.xo_encode_tile_m1.argtypes = [C.c_void_p, u64, u64, u64, C.c_int, C.c_void_p]
        L.xo_encode_tile_m2.restype = u64
        L.xo_encode_tile_m2.argtypes = [C.c_void_p, u64, u64, u64, C.c_void_p]
        L.xo_encode.restype = u64
        L.xo_encode.argtypes = [C.c_int, C.c_void_p, u64, u64, C.c_int, C.c_void_p]
        L.xo_peek.restype = C.c_int
        L.xo_peek.argtypes = [C.c_void_p, u64, C.POINTER(u64), C.POINTER(u64), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.xo_decode.restype = C.c_int
        L.xo_decode.argtypes = [C.c_void_p, u64, C.c_void_p]
        L.xo_trace.restype = None
        L.xo_trace.argtypes = [C.c_void_p, u64]
        L.xo_trace_len.restype = u64
        L.xo_trace_len.argtypes = []
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def tile_grid(w, h, pxsz=3):
    n = lib().xo_tile_grid(w, h, pxsz, None, 0)
    t = np.zeros((n, 4), dtype=np.uint64)
    lib().xo_tile_grid(w, h, pxsz, _ptr(t), n)
    return t  # rows: x, y, w, h


def normalize(px):
    px = np.ascontiguousarray(px, dtype=np.uint8)
    h, w, c = px.shape
    out = np.empty(h * w * c, dtype=np.uint8)
    s = C.c_uint64()
    a = lib().xo_normalize(_ptr(px), w, h, int(c == 4), _ptr(out), C.byref(s))
    return out[: s.value].reshape(h, w, 3 + a).copy()


def encode(mode, px):
    """(h,w,3|4) uint8 -> .xpng file bytes; raises on validation failure."""
    px = np.ascontiguousarray(px, dtype=np.uint8)
    h, w, c = px.shape
    out = np.empty(8 + h * w * c, dtype=np.uint8)
    n = lib().xo_encode(int(mode), _ptr(px), w, h, int(c == 4), _ptr(out))
    if n == 0:
        raise ValueError("oracle: encode rejected the input")
    return out[:n].tobytes()


# Decision log (xpng_oracle.h xo_trace): one record per size comparison of the encoder.
DECISION = np.dtype([("kind", "<u4"), ("tile", "<u4"), ("stream", "<u4"), ("outcome", "<u4"), ("v", "<u8", (4,))])
D_T1_TILE, D_FILE, D_T2_TILE, D_GREY_PLANE, D_GREY_PICK, D_V2_BLOCK, D_V2_TABLE, D_V1_BLOCK, D_V1_TABLE, D_PRED, D_STEAL = \
    range(1, 12)


def encode_traced(mode, px):
    """encode() with the decision log on: (file bytes, structured array of DECISION records in decision order)."""
    cap = 4096
    while True:
        buf = np.zeros(cap, dtype=DECISION)
        lib().xo_trace(_ptr(buf), cap)
        try:
            data = encode(mode, px)
            n = lib().xo_trace_len()
        finally:
            lib().xo_trace(None, 0)
        if n <= cap:
            return data, buf[:n].copy()
        cap = int(n)


def peek(data):
    buf = np.frombuffer(data, dtype=np.uint8)
    w, h, a, m = C.c_uint64(), C.c_uint64(), C.c_int(), C.c_int()
    rc = lib().xo_peek(_ptr(buf), len(buf), C.byref(w), C.byref(h), C.byref(a), C.byref(m))
    if rc:
        raise ValueError("oracle: bad header")
    return w.value, h.value, a.value, m.value


def decode(data):
    """.xpng bytes -> (h,w,3|4) uint8."""
    w, h, a, _ = peek(data)
    buf = np.frombuffer(bytes(data) + b"\0" * 16, dtype=np.uint8)
    out = np.zeros((h, w, 3 + a), dtype=np.uint8)
    if lib().xo_decode(_ptr(buf), len(data), _ptr(out)):
        raise ValueError("oracle: decode failed")
    return out


def select_predictor(img, x, y, w, h):
    H, W, c = img.shape
    base = img.ctypes.data + (y * W + x) * c
    return lib().xo_select_predictor(C.c_void_p(base), w, h, W * c, c)


def m1_front(img, x, y, w, h, pr):
    """Mode-1 front end of one tile: (streams list of 10 arrays, F[512], k words)."""
    H, W, c = img.shape
    base = img.ctypes.data + (y * W + x) * c
    streams = np.zeros(2 * w * h + 16, dtype=np.uint8)
    lens = (C.c_uint32 * 10)()
    F = np.zeros(512, dtype=np.uint32)
    k = np.zeros(w * h + 8, dtype=np.uint32)
    nk = lib().xo_m1_front(C.c_void_p(base), w, h, W * c, c, pr, _ptr(streams), lens,
                           F.ctypes.data_as(C.POINTER(C.c_uint32)), _ptr(k))
    out, off = [], 0
    for i in range(10):
        out.append(streams[off: off + lens[i]].copy())
        off += lens[i]
    return out, F, k[:nk].copy()


# ---------------------------------------------------------------- .7 container (7/libseven.c:3-36)

def write_7(path, px):
    px = np.ascontiguousarray(px, dtype=np.uint8)
    h, w, c = px.shape
    hdr = np.array([(w - 1) | (7 << 24), (h - 1) | ((c - 3) << 24)], dtype="<u4")
    with open(path, "wb") as f:
        f.write(hdr.tobytes())
        f.write(px.tobytes())


def read_7(path):
    raw = open(path, "rb").read()
    hdr = np.frombuffer(raw[:8], dtype="<u4")
    w, h, a = int(hdr[0] & 0xFFFFFF) + 1, int(hdr[1] & 0xFFFFFF) + 1, int(hdr[1] >> 24) & 1
    assert (hdr[0] >> 24) == 7 and len(raw) == 8 + w * h * (3 + a)
    return np.frombuffer(raw[8:], dtype=np.uint8).reshape(h, w, 3 + a).copy()


# ---------------------------------------------------------------- unmodified reference (oracle/_ref)

def ref_available():
    return os.path.exists(REF_CLI)


def _tmpdir():
    return "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()


def ref_encode(mode, px, cli=REF_CLI):
    """Run the reference CLI: .7 -> .xpng bytes (None if the reference fails or crashes)."""
    with tempfile.TemporaryDirectory(dir=_tmpdir()) as d:
        src, dst = os.path.join(d, "a.7"), os.path.join(d, "a.xpng")
        write_7(src, px)
        r = subprocess.run([cli, "-%d" % mode, src, dst], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        if r.returncode != 0 or not os.path.exists(dst):
            return None
        return open(dst, "rb").read()


def ref_decode(data, cli=REF_CLI):
    with tempfile.TemporaryDirectory(dir=_tmpdir()) as d:
        src, dst = os.path.join(d, "a.xpng"), os.path.join(d, "a.7")
        open(src, "wb").write(data)
        r = subprocess.run([cli, "-d", src, dst], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        if r.returncode != 0:
            return None
        return read_7(dst)


# ---------------------------------------------------------------------------------------------------------------
# Traversal-order operations (Mirroring_and_Rotating/tool.c) restated in numpy; test infrastructure like the rest.
REF_TOOL = os.path.join(_REF_DIR, "tool")
TOOL_OPS = ("r90", "r270", "mv", "mh", "mvh", "tl", "tr")          # option table, tool.c:133


def orient(op, px):
    """What `tool --<op>` leaves in the .7 file for pixmap px (h,w,c)."""
    if op == "mv":       # op_mv, tool.c:3-26: rows swapped top <-> bottom
        return px[::-1].copy()
    if op == "mh":       # op_mh, tool.c:28-59: pixels of every row reversed
        return px[:, ::-1].copy()
    if op == "mvh":      # op_mvh, tool.c:61-90: both (a half turn)
        return px[::-1, ::-1].copy()
    if op == "r90":      # op_r90, tool.c:92-112: src(i,j) -> dst(j, h-1-i), a clockwise quarter turn
        return np.ascontiguousarray(np.rot90(px, k=-1))
    if op == "r270":     # op_r270, tool.c:114-119: op_mvh then op_r90
        return np.ascontiguousarray(np.rot90(px[::-1, ::-1], k=-1))
    if op in ("tl", "tr"):   # op_tl / op_tr, tool.c:121-127: empty bodies
        return px.copy()
    raise ValueError(op)


def ref_orient(op, px):
    """The unmodified reference tool on a .7 file (oracle/_ref/tool)."""
    with tempfile.TemporaryDirectory(dir=_tmpdir()) as d:
        a, b = os.path.join(d, "s.7"), os.path.join(d, "x.7")
        write_7(a, px)
        subprocess.run([REF_TOOL, "--" + op, a, b], check=True, stdout=subprocess.DEVNULL)
        return read_7(b)
