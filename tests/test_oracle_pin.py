"""Pins the CPU oracle (oracle/xpng_oracle.c) to the unmodified reference:
 * against the committed golden manifest (sha256 of files the reference produced, tools/make_golden.py),
 * against the stored results of the reference on random inputs (tests/golden/reference_pins.json),
 * and, when oracle/_ref is present, directly against the reference binary on those inputs.
CPU only."""
import numpy as np
import pytest

from conftest import all_cases, make_case, reference_pins, sha
from oracle import pyoracle as po
from xpng_b200 import synth


@pytest.mark.parametrize("group,name,entry", all_cases(), ids=lambda v: v if isinstance(v, str) else "")
def test_oracle_matches_golden(group, name, entry):
    px = make_case(group, name, entry)
    assert list(px.shape) == entry["shape"]
    for lv in (1, 2, 7):
        f = po.encode(lv, px)
        assert len(f) == entry["levels"][str(lv)]["size"], (name, lv)
        assert sha(f) == entry["levels"][str(lv)]["sha256"], (name, lv)
        back = po.decode(f)
        assert list(back.shape) == entry["decoded_shape"]
        assert sha(back.tobytes()) == entry["decoded_sha256"]


@pytest.mark.parametrize("group,name,entry", all_cases(("corpus",)), ids=lambda v: v if isinstance(v, str) else "")
def test_oracle_matches_golden_corpus(group, name, entry):
    test_oracle_matches_golden(group, name, entry)


@pytest.mark.slow
@pytest.mark.parametrize("name", ["rgb_4k_s1", "gray_4096_s3000"])
def test_oracle_matches_golden_full_size(name):
    from conftest import manifest
    e = manifest()["synthetic"][name]
    test_oracle_matches_golden("synthetic", name, e)


def random_case(seed):
    """Input of test_oracle_matches_reference_binary for one seed (also read by tools/make_golden_pins.py)."""
    rng = np.random.default_rng(100 + seed)
    h, w = int(rng.integers(5, 700)), int(rng.integers(5, 900))
    gen = [synth.rgb, synth.rgba, synth.gray_as_rgb][seed % 3]
    return gen(h, w, 500 + seed)


@pytest.mark.parametrize("seed", range(6))
def test_oracle_matches_reference_binary(seed):
    """The oracle against the reference encoder and decoder on random shapes: against what the reference produced for these
    inputs (tests/golden/reference_pins.json) always, and against the reference binary itself when oracle/_ref is built."""
    px = random_case(seed)
    pin = reference_pins()["oracle_vs_reference"][str(seed)]
    assert list(px.shape) == pin["shape"]
    for lv in (1, 2, 7):
        a = po.encode(lv, px)
        back = po.decode(a)
        assert len(a) == pin[str(lv)]["size"] and sha(a) == pin[str(lv)]["sha256"], lv
        assert list(back.shape) == pin["decoded_shape"] and sha(back.tobytes()) == pin[str(lv)]["decoded_sha256"], lv
        if po.ref_available():
            assert a == po.ref_encode(lv, px)
            assert np.array_equal(back, po.ref_decode(a))


def test_tile_grid_baseline_shapes():
    """SURVEY §8: 4K -> 9x5, 1080p -> 4x2, 8192^2 -> 18x18, 4096^2 -> 9x9 tiles."""
    assert len(po.tile_grid(3840, 2160)) == 45
    t = po.tile_grid(1920, 1080)
    assert len(t) == 8 and sorted(set(t[:, 2].tolist())) == [444, 588] and sorted(set(t[:, 3].tolist())) == [444, 636]
    assert len(po.tile_grid(8192, 8192, 4)) == 324
    assert len(po.tile_grid(4096, 4096)) == 81
    for (w, h) in [(3840, 2160), (1334, 750), (37, 1500), (1500, 37), (445, 445), (1, 1), (667, 889)]:
        t = po.tile_grid(w, h)
        assert int((t[:, 2] * t[:, 3]).sum()) == w * h


def test_rgba_tiny_is_rejected():
    """The reference crashes on RGBA tiles thinner than 4 (SURVEY App. C.1); we fail cleanly."""
    with pytest.raises(ValueError):
        px = synth.rgb(5, 3, 1, channels=4); px[..., 3] = 128
        po.encode(1, px)


def test_ycocg_r_exhaustive():
    """Tell_Me_Why/YCoCg-R.c: lifting is reversible over all 2^24 triples, Co/Cg in [-255,255]."""
    r, g, b = np.meshgrid(np.arange(256), np.arange(256), np.arange(256), indexing="ij")
    co = r - b; t = b + (co >> 1); cg = g - t; y = t + (cg >> 1)
    assert y.min() == 0 and y.max() == 255 and co.min() == -255 and co.max() == 255 and cg.min() == -255 and cg.max() == 255
    t2 = y - (cg >> 1); g2 = cg + t2; b2 = t2 - (co >> 1); r2 = b2 + co
    assert np.array_equal(r, r2) and np.array_equal(g, g2) and np.array_equal(b, b2)
