"""Traversal-order operations (SURVEY §8 f3; reference Mirroring_and_Rotating/tool.c).
CPU: the numpy restatement in oracle/pyoracle.py against the unmodified reference tool (its stored outputs, and
oracle/_ref/tool when built) and the reference's own reversibility.rb properties.  GPU: k_orient through the C ABI against the restatement, the encoder's
orientation option against "tool then xpng" of the oracle, and the `tool` command line."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, reference_pins, sha
from oracle import pyoracle as po
from xpng_b200 import synth

TOOL = os.path.join(ROOT, "xpng_b200", "bin", "tool")
SHAPES = [(1, 1, 3), (1, 7, 3), (9, 1, 4), (5, 3, 4), (64, 64, 3), (65, 63, 4), (100, 257, 3), (311, 129, 4), (200, 130, 3)]


def _px(shape, seed=5):
    return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)


@pytest.mark.parametrize("op", po.TOOL_OPS)
def test_restatement_matches_reference_tool(op):
    """Against what the reference tool wrote for these inputs (tests/golden/reference_pins.json) always, and against the tool
    itself when oracle/_ref is built."""
    pins = reference_pins()["orient"][op]
    for shape in SHAPES:
        px = _px(shape)
        got = po.orient(op, px)
        want_shape, want_sha = pins["x".join(map(str, shape))]
        assert list(got.shape) == want_shape and sha(got.tobytes()) == want_sha, (op, shape)
        if os.path.exists(po.REF_TOOL):
            assert np.array_equal(got, po.ref_orient(op, px)), (op, shape)


def test_restatement_reversibility():
    """reversibility.rb:12-19: r90 then r270 is the identity, every other op is an involution."""
    for shape in SHAPES:
        px = _px(shape, 6)
        assert np.array_equal(po.orient("r270", po.orient("r90", px)), px)
        for op in ("mv", "mh", "mvh", "tl", "tr"):
            assert np.array_equal(po.orient(op, po.orient(op, px)), px)


@pytest.fixture(scope="module")
def codec():
    import xpng_b200
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


@pytest.mark.gpu
@pytest.mark.parametrize("op", po.TOOL_OPS)
def test_transform_matches_restatement(codec, op):
    imgs = [_px(s, 7 + i) for i, s in enumerate(SHAPES)] + [synth.rgb(1080, 1920, 3), synth.rgba(700, 901, 4)]
    got = codec.transform(op, imgs)            # one batched launch
    for g, im in zip(got, imgs):
        want = po.orient(op, im)
        assert g.shape == want.shape and np.array_equal(g, want), (op, im.shape)


@pytest.mark.gpu
def test_transform_reversibility_on_device(codec):
    imgs = [synth.rgb(500, 333, 1), synth.rgba(222, 444, 2)]
    back = codec.transform("r270", codec.transform("r90", imgs))
    assert all(np.array_equal(a, b) for a, b in zip(back, imgs))
    for op in ("mv", "mh", "mvh", "tl", "tr"):
        back = codec.transform(op, codec.transform(op, imgs))
        assert all(np.array_equal(a, b) for a, b in zip(back, imgs)), op


@pytest.mark.gpu
@pytest.mark.parametrize("level", (1, 2, 7))
def test_encode_oriented_equals_tool_then_encode(codec, level):
    """Mirroring_and_Rotating/test.rb: every orientation of an image encoded; files must equal the oracle's."""
    imgs = [synth.rgb(600, 911, 11), synth.rgba(450, 300, 12), synth.gray_as_rgb(333, 500, 13)]
    for op in po.TOOL_OPS:
        got = codec.encode_oriented(level, op, imgs)
        for g, im in zip(got, imgs):
            assert g == po.encode(level, po.orient(op, im)), (op, level, im.shape)
        back = codec.decode(got)
        for b, im in zip(back, imgs):
            assert np.array_equal(b, po.normalize(po.orient(op, im)))


@pytest.mark.gpu
def test_tool_cli(tmp_path):
    px = synth.rgba(123, 77, 9)
    src, dst = str(tmp_path / "s.7"), str(tmp_path / "x.7")
    po.write_7(src, px)
    for op in po.TOOL_OPS:
        assert subprocess.run([TOOL, "--" + op, src, dst]).returncode == 0
        assert np.array_equal(po.read_7(dst), po.orient(op, px)), op
    # in place, like test.rb:35 (`tool --r90 /tmp/s.7 /tmp/s.7`)
    assert subprocess.run([TOOL, "--r90", src, src]).returncode == 0
    assert np.array_equal(po.read_7(src), po.orient("r90", px))


def test_tool_cli_usage(tmp_path):
    """tool.c:129-141: wrong argument count or option name -> usage text, exit 1; unreadable input -> exit 1, silent."""
    want = "\n\t./tool --(r90|r270|mv|mh|mvh|tl|tr) src.7 res.7\n\n"
    r = subprocess.run([TOOL], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == want
    src = str(tmp_path / "s.7")
    po.write_7(src, _px((4, 4, 3)))
    r = subprocess.run([TOOL, "--flip", src, str(tmp_path / "o.7")], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == want
    r = subprocess.run([TOOL, "--mv", str(tmp_path / "missing.7"), str(tmp_path / "o.7")], capture_output=True, text=True)
    assert r.returncode == 1 and r.stdout == ""
    if os.path.exists(po.REF_TOOL):
        for args in ([], ["--flip", src, "/dev/null"], ["--mv", str(tmp_path / "missing.7"), "/dev/null"]):
            a = subprocess.run([po.REF_TOOL] + args, capture_output=True, text=True)
            b = subprocess.run([TOOL] + args, capture_output=True, text=True)
            assert (a.returncode, a.stdout) == (b.returncode, b.stdout), args
