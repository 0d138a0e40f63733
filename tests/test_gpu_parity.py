"""GPU parity tests proper (B200): the CUDA path, called through the C ABI, against the CPU oracle,
the committed golden manifest (sha256 of files written by the unmodified reference) and, when it
travelled with the snapshot, the reference binary itself.  Bit-exact everywhere (integer codec)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, all_cases, make_case, manifest, reference_pins, sha
from oracle import pyoracle as po
from xpng_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def codec():
    import xpng_b200
    cd = xpng_b200.Codec(0)
    yield cd
    cd.close()


@pytest.mark.parametrize("group,name,entry", all_cases(("synthetic", "special", "crops", "corpus"), big=True),
                         ids=lambda v: v if isinstance(v, str) else "")
def test_golden_bytes_and_roundtrip(codec, group, name, entry):
    px = make_case(group, name, entry)
    for lv in (1, 2, 7):
        f = codec.encode(lv, [px])[0]
        assert len(f) == entry["levels"][str(lv)]["size"], (name, lv)
        assert sha(f) == entry["levels"][str(lv)]["sha256"], (name, lv)
        back = codec.decode([f])[0]
        assert list(back.shape) == entry["decoded_shape"]
        assert sha(back.tobytes()) == entry["decoded_sha256"], (name, lv)


@pytest.mark.parametrize("seed", range(12))
def test_random_shapes_against_oracle(codec, seed):
    rng = np.random.default_rng(1000 + seed)
    h, w = int(rng.integers(4, 1200)), int(rng.integers(4, 1400))
    gen = [synth.rgb, synth.rgba, synth.gray_as_rgb, synth.noise][seed % 4]
    px = gen(h, w, 700 + seed)
    for lv in (1, 2, 7):
        want = po.encode(lv, px)
        got = codec.encode(lv, [px])[0]
        assert got == want, (h, w, lv)
        assert np.array_equal(codec.decode([want])[0], po.normalize(px))


def test_batch_mixed_shapes(codec):
    """Several images of different shapes / alpha in one call: every file equals the single-image oracle file."""
    imgs = [synth.rgb(300 + 37 * i, 500 + 91 * i, 40 + i) for i in range(5)] + [synth.rgba(400, 333, 50), synth.gray_as_rgb(200, 700, 51),
            np.full((64, 64, 3), 9, np.uint8), synth.rgb(1, 1, 3)]
    for lv in (1, 2, 7):
        got = codec.encode(lv, imgs)
        assert got == [po.encode(lv, im) for im in imgs]
        back = codec.decode(got)
        for b, im in zip(back, imgs):
            assert np.array_equal(b, po.normalize(im))


def test_frame_sequence_config3(codec):
    """BASELINE config 3 in small: a batch of 1080p 'sintel-like' frames, level 1 and 2."""
    frames = [synth.sintel_like(1000 + i) for i in range(6)]
    man = manifest()["synthetic"]
    for lv in (1, 2):
        files = codec.encode(lv, frames)
        assert sha(files[0]) == man["sintel_1080p_s1000"]["levels"][str(lv)]["sha256"]
        assert sha(files[1]) == man["sintel_1080p_s1001"]["levels"][str(lv)]["sha256"]
        for f, fr in zip(files, frames):
            assert f == po.encode(lv, fr)
        for b, fr in zip(codec.decode(files), frames):
            assert np.array_equal(b, fr)


def test_rgba_tiny_is_rejected(codec):
    px = synth.rgb(5, 3, 1, channels=4); px[..., 3] = 128
    with pytest.raises(RuntimeError):
        codec.encode(1, [px])
    assert len(codec.encode(7, [px])[0]) == 8 + px.size      # stored is fine


def test_corrupt_input_fails_cleanly(codec):
    f = bytearray(po.encode(1, synth.rgb(300, 300, 5)))
    f[9] ^= 0xFF; f[10] ^= 0x7F        # first tile's size field
    with pytest.raises(RuntimeError):
        codec.decode([bytes(f)])
    with pytest.raises((RuntimeError, ValueError)):
        codec.decode([b"\0" * 16])


def test_device_resident_buffers(codec):
    """Device pointers in, device pointers out (what bench.py times as `value`)."""
    import torch
    import xpng_b200
    frames = [synth.rgb(720, 1280, 60 + i) for i in range(3)]
    descs, total = xpng_b200.Codec.layout([f.shape for f in frames])
    host = np.zeros(total, np.uint8)
    for d, f in zip(descs, frames):
        host[d.offset: d.offset + f.size] = f.reshape(-1)
    dpx = torch.from_numpy(host).cuda()
    cap = int(xpng_b200.lib().xpngb_encode_bound(descs, 3))
    dout = torch.empty(cap, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    offs, sizes = codec.encode_raw(1, descs, 3, dpx.data_ptr(), total, 1, dout.data_ptr(), cap, 1)
    out = dout.cpu().numpy()
    files = [out[offs[i]: offs[i] + sizes[i]].tobytes() for i in range(3)]
    assert files == [po.encode(1, f) for f in frames]
    dback = torch.zeros(total, dtype=torch.uint8, device="cuda")
    for d in descs:
        d.w = d.h = 0   # let the decoder fill them from the headers
    codec.decode_raw(descs, 3, dout.data_ptr(), cap, 1, offs, sizes, dback.data_ptr(), total, 1)
    assert np.array_equal(dback.cpu().numpy(), host)


CLI_CASES = {"rgb_333x517_s8": (synth.rgb, 333, 517, 8), "rgba_250x300_s9": (synth.rgba, 250, 300, 9)}


def test_file_api_and_cli_against_reference(codec, tmp_path):
    """xpng_store / xpng_load (xpng.h) and the CLI contract of xpng.c / test.rb: .7 -> .xpng -> .7 + cmp.  The files must be
    the reference's (tests/golden/reference_pins.json; the reference binary decodes them too when oracle/_ref is built)."""
    import xpng_b200
    cli = os.path.join(ROOT, "xpng_b200", "bin", "xpng")
    pins = reference_pins()["file_api_cli"]
    for key, (gen, h, w, seed) in CLI_CASES.items():
        px = gen(h, w, seed)
        src = str(tmp_path / "src.7"); po.write_7(src, px)
        for lv in (1, 2, 7):
            dst, back = str(tmp_path / "res.xpng"), str(tmp_path / "res.7")
            r = subprocess.run([cli, f"-{lv}", src, dst], capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            assert open(dst, "rb").read() == po.encode(lv, px)
            assert sha(open(dst, "rb").read()) == pins[key][str(lv)], (key, lv)
            if lv != 7:
                assert r.stdout.startswith("encode,") and r.stdout.rstrip().endswith("MPx/s")   # libxpng.c:761
            r = subprocess.run([cli, "-d", dst, back], capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            assert np.array_equal(po.read_7(back), po.normalize(px))
            # library entry points directly
            assert xpng_b200.xpng_store(lv, px, dst) is False
            assert open(dst, "rb").read() == po.encode(lv, px)
            assert np.array_equal(xpng_b200.xpng_load(dst), po.normalize(px))
            if po.ref_available():   # the unmodified reference decodes our file, and we decode its file
                assert np.array_equal(po.ref_decode(open(dst, "rb").read()), po.normalize(px))
                assert np.array_equal(codec.decode([po.ref_encode(lv, px)])[0], po.normalize(px))


def test_file_api_is_reentrant(codec, tmp_path):
    """xpng_store / xpng_load from several host threads at once (the reference keeps no global mutable state, SURVEY 8(b)):
    every caller takes its own codec context from the library's pool; results equal the oracle's."""
    import xpng_b200
    from concurrent.futures import ThreadPoolExecutor
    imgs = [synth.rgb(200 + 37 * k, 300 + 11 * k, 90 + k) for k in range(6)] + [synth.rgba(180, 260, 97)]

    def job(k):
        px, lv, fn = imgs[k], 1 + (k & 1), str(tmp_path / f"t{k}.xpng")
        for _ in range(3):
            assert xpng_b200.xpng_store(lv, px, fn) is False
            assert open(fn, "rb").read() == po.encode(lv, px)
            assert np.array_equal(xpng_b200.xpng_load(fn), po.normalize(px))
        return True

    with ThreadPoolExecutor(len(imgs)) as pool:
        assert all(pool.map(job, range(len(imgs))))


def test_ycocg_r_side_kernel(codec):
    """Tell_Me_Why/YCoCg-R.c: exhaustive 2^24 reversibility and ranges, on the device."""
    r, g, b = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
    rgb = np.stack([r, g, b], axis=-1).reshape(-1, 3)
    ycc = codec.ycocg_forward(rgb)
    assert ycc[:, 0].min() == 0 and ycc[:, 0].max() == 255
    assert ycc[:, 1].min() == -255 and ycc[:, 1].max() == 255 and ycc[:, 2].min() == -255 and ycc[:, 2].max() == 255
    assert np.array_equal(codec.ycocg_inverse(ycc), rgb)


def test_throughput_kernel_family(monkeypatch):
    """Large batches switch from the warp-per-block (latency) entropy kernels to the lane-per-block ones
    (XPNGB_LAT_MAX_BLOCKS, read when the context is created): both families must produce the same bytes."""
    import xpng_b200
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    cd = xpng_b200.Codec(0)
    try:
        imgs = [synth.rgb(500, 700, 81), synth.rgba(450, 460, 82), synth.gray_as_rgb(300, 520, 83), synth.noise(90, 70, 84),
                np.full((50, 60, 3), 7, np.uint8)]
        for lv in (1, 2):
            want = [po.encode(lv, im) for im in imgs]
            assert cd.encode(lv, imgs) == want
            for b, im in zip(cd.decode(want), imgs):
                assert np.array_equal(b, po.normalize(im))
        # corrupt files through this family as well: failure or garbage, never a fault
        rng = np.random.default_rng(11)
        for lv, img in ((1, imgs[1]), (2, imgs[0])):
            good = po.encode(lv, img)
            for k in range(16):
                f = bytearray(good)
                for _ in range(int(rng.integers(1, 6))):
                    f[int(rng.integers(8, len(f)))] = int(rng.integers(0, 256))
                try:
                    cd.decode([bytes(f)])
                except RuntimeError:
                    pass
            assert np.array_equal(cd.decode([good])[0], po.normalize(img))
    finally:
        cd.close()


def test_batch_decode_variants(monkeypatch):
    """Decode variants that batches select by residency (ring-staged context walk, two-level tables for every level-2
    block), forced here on small inputs: same pixels, and corrupt files neither fault nor poison the context."""
    import xpng_b200
    monkeypatch.setenv("XPNGB_WALK", "ring")
    monkeypatch.setenv("XPNGB_DIRECT_MAX_TILES", "0")
    cd = xpng_b200.Codec(0)
    try:
        imgs = [synth.rgb(700, 900, 91), synth.rgba(450, 460, 92), synth.gray_as_rgb(300, 520, 93), synth.noise(90, 70, 94),
                synth.rgb(5, 2000, 95), synth.sintel_like(1003)]
        for lv in (1, 2):
            want = [po.encode(lv, im) for im in imgs]
            for b, im in zip(cd.decode(want), imgs):
                assert np.array_equal(b, po.normalize(im)), (lv, im.shape)
        rng = np.random.default_rng(12)
        for lv, img in ((1, imgs[1]), (2, imgs[0]), (1, imgs[5])):
            good = po.encode(lv, img)
            for k in range(24):
                f = bytearray(good)
                for _ in range(int(rng.integers(1, 6))):
                    f[int(rng.integers(8, len(f)))] = int(rng.integers(0, 256))
                try:
                    cd.decode([bytes(f)])
                except RuntimeError:
                    pass
            assert np.array_equal(cd.decode([good])[0], po.normalize(img))
    finally:
        cd.close()


def test_largest_tile_uses_ring_walk(codec):
    """A 666 x 666 image is ONE tile (libxpng.c:57-80) of 443 556 pixels: its context streams do not fit the
    shared-memory walk, so the ring-staged walk (k_dec_walk_ring) runs instead."""
    px = synth.rgb(666, 666, 91)
    for lv in (1, 2):
        want = po.encode(lv, px)
        assert codec.encode(lv, [px])[0] == want
        assert np.array_equal(codec.decode([want])[0], px)


def test_many_small_images_one_call(codec):
    """More than 592 tiles in one call (4 tiles per CTA variants of the per-tile kernels)."""
    imgs = [synth.rgb(20 + (i % 7), 24 + (i % 5), 2000 + i) for i in range(640)]
    for lv in (1, 2):
        want = [po.encode(lv, im) for im in imgs]
        assert codec.encode(lv, imgs) == want
        for b, im in zip(codec.decode(want), imgs):
            assert np.array_equal(b, im)


def test_fuzzed_files_never_crash(codec):
    """Random byte corruption of valid files: the decoder may fail (RuntimeError) or return garbage, but it must
    neither hang nor fault (a CUDA fault would poison the context and fail the final clean decode)."""
    rng = np.random.default_rng(7)
    px = synth.rgba(300, 340, 93)
    rgbpx = synth.rgb(320, 300, 94)
    for lv, img in ((1, px), (1, rgbpx), (2, rgbpx), (2, synth.gray_as_rgb(200, 260, 95))):
        good = po.encode(lv, img)
        for k in range(24):
            f = bytearray(good)
            for _ in range(int(rng.integers(1, 6))):
                pos = int(rng.integers(8, len(f)))
                f[pos] = int(rng.integers(0, 256))
            try:
                codec.decode([bytes(f)])
            except RuntimeError:
                pass
        assert np.array_equal(codec.decode([good])[0], po.normalize(img))


def _level2_with_oversized_value_blocks(img):
    """A valid single-tile level-2 file whose eight value blocks (st1..st8, App. A.5) are replaced by type-1 runs that each
    claim 3 * npx symbols: every block passes a per-block bound, their sum is far beyond the tile's stream slice."""
    import struct
    f = po.encode(2, img)
    h, w = img.shape[:2]
    assert (struct.unpack_from("<I", f, 0)[0] >> 24) == 2
    t0 = 8
    tw = struct.unpack_from("<I", f, t0)[0]
    assert (tw >> 24) & 0xF0 == 0x10 and (tw & 0xFFFFFF) == len(f) - 8       # one coded RGB tile
    bsz = struct.unpack_from("<I", f, t0 + 4)[0]
    p = t0 + 4 + bsz                                                          # first of the 17 v1 blocks
    for _ in range(9):                                                        # keep the nine context blocks
        p += struct.unpack_from("<I", f, p)[0] & 0xFFFFFF
    body = bytearray(f[:p])
    for _ in range(8):                                                        # type 1: [8 | 1 << 24][n | sym << 24]
        body += struct.pack("<II", 8 | (1 << 24), (3 * w * h) | (5 << 24))
    struct.pack_into("<I", body, t0, (len(body) - 8) | (tw & 0xFF000000))
    return bytes(body)


def test_crafted_value_block_counts_are_rejected(codec):
    """ADVICE round 1 (high): the running stream offset of a level-2 tile must be bounded, not only each block."""
    img = synth.rgb(96, 128, 77)
    bad = _level2_with_oversized_value_blocks(img)
    for fam in ("0", "10000000"):                      # both decoder families
        os.environ["XPNGB_LAT_MAX_BLOCKS"] = fam
        try:
            import xpng_b200
            cd = xpng_b200.Codec(0)
            with pytest.raises(RuntimeError):
                cd.decode([bad])
            # the context is still healthy and nothing outside the tile's slice was written: a clean decode follows
            assert np.array_equal(cd.decode([po.encode(2, img)])[0], img)
            cd.close()
        finally:
            del os.environ["XPNGB_LAT_MAX_BLOCKS"]


def test_thin_tiles_first_in_batch(codec):
    """Regression (found by tools/parity_sweep.py): a 1-pixel-wide tile whose scratch slice starts the buffer must not
    read the word before its residual plane; thin and very wide tiles take different un-predict kernels."""
    batch = [synth.rgb(1823, 1, 5), synth.rgb(1, 1399, 6), synth.rgb(196, 393, 7), synth.rgba(9, 914, 8), synth.rgb(436, 3, 9)]
    for lv in (1, 2):
        want = [po.encode(lv, im) for im in batch]
        assert codec.encode(lv, batch) == want
        for b, im in zip(codec.decode(want), batch):
            assert np.array_equal(b, po.normalize(im))


def test_randomised_sweep(codec):
    """A slice of tools/parity_sweep.py (mixed batches of random shapes and content classes) on every run."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("parity_sweep", os.path.join(ROOT, "tools", "parity_sweep.py"))
    ps = importlib.util.module_from_spec(spec); spec.loader.exec_module(ps)
    rng = np.random.default_rng(31337)
    for _ in range(20):
        batch = [ps.make(rng, []) for _ in range(int(rng.integers(1, 6)))]
        for lv in (1, 2, 7):
            want = [po.encode(lv, im) for im in batch]
            assert codec.encode(lv, batch) == want, [im.shape for im in batch]
            for b, im in zip(codec.decode(want), batch):
                assert np.array_equal(b, po.normalize(im)), im.shape


def test_config3_golden_64_frames_pipelined(monkeypatch):
    """BASELINE configs[2], the first 64 frames, against files written by the unmodified reference
    (tests/golden/config3_64.json, tools/make_golden_config3.py).  The call is forced through the batch machinery:
    several chunks on concurrent lanes (XPNGB_PIPE_MIN_MPIX), the pair-lane rANS kernels, the sorted work lists and
    the three-tiles-per-warp walk (XPNGB_LAT_MAX_BLOCKS=0)."""
    import hashlib
    import json
    import xpng_b200
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "config3_64.json")))
    frames = synth.sintel_batch(range(1000, 1064))
    monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    monkeypatch.setenv("XPNGB_PIPE_MIN_MPIX", "20")
    monkeypatch.setenv("XPNGB_PIPE_LANES", "4")      # 7 chunks on 4 lanes: lanes are reused within the call
    cd = xpng_b200.Codec(0)
    try:
        for lv in (1, 2):
            files = cd.encode(lv, frames)
            for k, f in enumerate(files):
                size, digest = gold[str(1000 + k)][str(lv)]
                assert len(f) == size and hashlib.sha256(f).hexdigest() == digest, (lv, 1000 + k)
            for b, im in zip(cd.decode(files), frames):
                assert np.array_equal(b, im), lv
    finally:
        cd.close()


def test_dropin_relink_of_the_reference_cli(tmp_path):
    """The reference's own CLI source (xpng.c), compiled where it lies and linked against libxpng_b200.so instead of
    libxpng.c / libseven.c (oracle/Makefile: _ref/xpng_dropin): .7 -> .xpng -> .7 with files identical to the reference's."""
    dropin = os.path.join(ROOT, "oracle", "_ref", "xpng_dropin")
    if not os.path.exists(dropin):
        pytest.skip("oracle/_ref/xpng_dropin absent (built where /root/reference exists)")
    px = synth.rgb(300, 410, 77)
    src = str(tmp_path / "a.7"); po.write_7(src, px)
    for lv in (1, 2, 7):
        out, back = str(tmp_path / f"a{lv}.xpng"), str(tmp_path / f"b{lv}.7")
        assert subprocess.run([dropin, f"-{lv}", src, out], capture_output=True).returncode == 0
        assert open(out, "rb").read() == po.encode(lv, px)
        assert subprocess.run([dropin, "-d", out, back], capture_output=True).returncode == 0
        assert open(back, "rb").read() == open(src, "rb").read()


def test_sharded_pool_matches_one_device():
    """xpngb_pool_encode / xpngb_pool_decode (host threads, one context per device, no NCCL): the files and the size
    table of a batch cut over two devices equal those of one device."""
    import hashlib
    import torch
    from xpng_b200 import shard
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    frames = [synth.rgb(200 + 7 * i, 300 + 5 * i, 600 + i) for i in range(9)] + [synth.rgba(120, 90, 3)]
    shas = []
    for devs in ([0], [0, 1]):
        pool = shard.Pool(devs)
        try:
            for lv in (1, 2):
                files, offs, sizes = pool.encode(lv, frames)
                assert files == [po.encode(lv, f) for f in frames]
                shas.append((lv, hashlib.sha256(np.asarray(sizes, np.uint64).tobytes()).hexdigest()))
                for b, im in zip(pool.decode(files), frames):
                    assert np.array_equal(b, po.normalize(im))
        finally:
            pool.close()
    assert shas[:2] == shas[2:]


def test_single_device_pool_and_wide_one_tile_image():
    """A one-device pool is the plain codec; a 37-row image is ONE tile 1500 pixels wide, which the staged RGB front end
    leaves to the first-generation kernel."""
    from xpng_b200 import shard
    frames = [synth.rgb(37, 1500, 6), synth.rgb(1500, 37, 5), synth.rgb(64, 671, 9), synth.rgb(64, 670, 9)]
    pool = shard.Pool([0])
    try:
        for lv in (1, 2):
            files, offs, sizes = pool.encode(lv, frames)
            assert files == [po.encode(lv, f) for f in frames]
            for b, im in zip(pool.decode(files), frames):
                assert np.array_equal(b, im)
    finally:
        pool.close()
