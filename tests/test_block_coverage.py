"""Every coded-block kind through every decoder kernel variant, and proof that both were reached.

The decode path is chosen at run time by what a file holds (tile kinds, block types, table forms, alphabets) and by the
size of the call (kernel families, table forms, walks, un-predict kernels).  FEATURES is a small deterministic image set
whose oracle files hold every block kind in REQUIRED (checked by tests/xpng_walk.py, without a GPU); the GPU tests decode
it under each kernel configuration of decode_issue (csrc/api.cu) and assert both pixel parity with the CPU oracle and,
from the profile report, that the configuration's kernels ran.
"""
import os

import numpy as np
import pytest

from conftest import CORPUS, all_cases, load_png, make_case
from oracle import pyoracle as po
from xpng_b200 import synth
import xpng_walk as xw

LEVELS = (1, 2, 7)


# ---------------------------------------------------------------------------------------------------------------- images

def _grey(v):
    return np.repeat((np.asarray(v, dtype=np.int64) % 256).astype(np.uint8)[..., None], 3, axis=2)


def _split(left, right):
    """Two tiles side by side: 444 rows of 350 + 350 pixels (xo_tile_grid splits 700 into two 350-wide tiles)."""
    return np.ascontiguousarray(np.concatenate([left, right], axis=1))


def _specks(shape, bg, n, seed, delta):
    """A flat plane with n isolated specks: the context streams are one symbol plus a handful of others."""
    rng = np.random.default_rng(seed)
    px = np.empty(shape, np.uint8)
    px[...] = bg
    for _ in range(n):
        y, x = int(rng.integers(8, shape[0] - 8)), int(rng.integers(8, shape[1] - 8))
        px[y, x] = (px[y, x].astype(int) + delta) % 256
    return px


def _dots():
    """A grid of red -1 dots on a flat plane and one blue dot: the nl = 1 value stream is one symbol and one other."""
    px = np.full((444, 444, 3), 120, np.uint8)
    px[1::4, 1::4, 0] -= 1
    px[223, 225, 2] -= 1
    return px


def _slopes():
    """One row whose left differences are the same in every channel and step through -1, -2, 2, 4, ... 64: each
    level-2 value stream (nl = 1 .. 8) holds a single symbol, a run block."""
    v = np.cumsum(np.repeat([-1, -2, 2, 4, 8, 16, 32, 64], 40)) % 256
    return (np.stack([v, v + 50, v + 100], axis=1)[None] % 256).astype(np.uint8)


def _corpus(name):
    return np.ascontiguousarray(load_png(os.path.join(CORPUS, name))[:444, :444])


def _features():
    y, x = np.mgrid[0:300, 0:300]
    rng = np.random.default_rng(5)
    walk = np.random.default_rng(20)
    rgb = lambda a, b, c: np.stack([a % 256, b % 256, c % 256], axis=2).astype(np.uint8)
    yield "split_noise_smooth", _split(synth.noise(444, 350, 1), synth.rgb(444, 350, 2))            # raw tile in a coded file
    yield "split_grey_noise", _split(_grey(synth.noise(444, 350, 3)[..., 0]), synth.gray_as_rgb(444, 350, 4))   # grey raw
    yield "split_flat_smooth", _split(np.full((444, 350, 3), 61, np.uint8), synth.rgb(444, 350, 24))   # single-colour tile
    yield "grey_ramp", _grey(x + y)                                                   # grey run block
    yield "grey_rows", _grey(x + rng.integers(0, 256, (300, 1)))                      # grey pm 0
    yield "grey_cols", _grey(y + rng.integers(0, 256, (1, 300)))                      # grey pm 1
    yield "grey_plane", _grey(5 * x + 7 * y + rng.integers(0, 2, (300, 300)))         # grey pm 2
    yield "grey_quad", _grey((x * x + y * y) // 300)                                  # grey pm 3
    yield "grey_smooth", synth.gray_as_rgb(300, 300, 6)
    yield "grey_walk", _grey(np.cumsum(np.round(walk.laplace(0, 20, (444, 444))).astype(int), axis=1))   # dense grey table
    yield "rgb_rows", rgb(x + rng.integers(0, 256, (300, 1)), 2 * x, x // 3)
    yield "rgb_cols", rgb(y + rng.integers(0, 256, (1, 300)), 2 * y, y // 3)
    yield "rgb_plane", rgb(5 * x + 7 * y, 3 * x + 2 * y, x + 9 * y) + rng.integers(0, 2, (300, 300, 3)).astype(np.uint8)
    yield "specks", _specks((444, 444, 3), (40, 90, 200), 5, 7, (9, 0, 0))           # dominant context symbol
    yield "grey_specks", _specks((444, 444, 3), (77, 77, 77), 5, 8, (30, 30, 30))    # dominant grey symbol
    yield "dots", _dots()                                                             # dominant value symbol
    yield "slopes", _slopes()
    yield "alpha_noise", np.concatenate([synth.rgb(300, 300, 10), rng.integers(1, 255, (300, 300, 1)).astype(np.uint8)], axis=2)
    yield "alpha_flat", np.concatenate([synth.rgb(200, 200, 11), np.full((200, 200, 1), 128, np.uint8)], axis=2)
    yield "alpha_specks", np.concatenate([synth.rgb(300, 300, 12), _specks((300, 300, 1), 200, 3, 13, 50)], axis=2)
    yield "flat", np.full((64, 80, 3), 33, np.uint8)                                  # single-colour file
    yield "noise", synth.noise(100, 120, 22)                                          # level-7 fallback
    yield "wide", synth.rgb(37, 1500, 23)                                             # one tile wider than 672
    for name in ("idiocracy.png", "Can_I_use_WebP_06-07-2022.png", "do_not_resist_intuition.png", "juicy.png", "body_shop.png"):
        yield "corpus_" + name, _corpus(name)                                       # large alphabets, sharp edges


FEATURES = list(_features())

# ------------------------------------------------------------------------------------------------ required features

_RANS = ("odd_n", "tail", "words>512", "w1")
REQUIRED = (
    {("file", f) for f in ("stored", "fallback7", "single", "m1", "m2")}
    | {("t1", f) for f in ("raw", "pr0", "pr1", "pr2", "pr3")}
    | {("t2", f) for f in ("raw", "single", "grey_raw", "grey_pm0", "grey_pm1", "grey_pm2", "grey_pm3", "pr0", "pr1", "pr2", "pr3")}
    | {("v2ctx", f) for f in ("type0", "type1", "type2", "type3", "type4", "dominant") + _RANS}
    | {("v2alpha", f) for f in ("type1", "type2", "type3", "type4", "dominant") + _RANS}
    | {("v1ctx", f) for f in ("type0", "type1", "type2", "type3", "type4", "dominant") + _RANS}
    | {(f"v1val{n}", f) for n in (8, 16, 32, 64, 128, 256) for f in ("type0", "type1", "type2", "type3", "type4") + _RANS}
    | {("v1val8", "dominant")}
    | {("v1grey", f) for f in ("type1", "type3", "type4", "dominant") + _RANS}
)

# What the reference encoder cannot write (xpng_oracle.c), with the reason; test_unreachable_features checks each claim.
UNREACHABLE = {
    ("v2alpha", "type0"): "an RGBA file needs w, h >= 4 (xo_encode) and tiles are at least that large, so the alpha block "
                          "holds npx - 1 >= 15 symbols",
    ("v1grey", "type0"): "n = npx - 1 is 0 only for a 1-pixel tile; a 1-pixel image is 3 bytes, stored (s <= 4), and a tile "
                         "of a larger image is at least half the base tile on each side",
    ("v1grey", "type2"): "raw grey symbols cost 8 bits each, so bsz + rsz >= 4 + 1 + npx - 1 + 8 > npx and encode_tile_grey "
                         "writes the grey plane raw instead",
    "n<32": "a rANS block of fewer than 32 symbols is never smaller than its raw form (checked for every alphabet and pb "
            "by test_rans_never_wins_below_32_symbols)",
}
# Reachable but not required: a dominant symbol in the 16- to 256-symbol value streams (nl >= 4 puts one symbol per
# channel into the stream, so a plane with a few specks does not make one symbol take all but 4 slots).

# ------------------------------------------------------------------------------------------------------- CPU tests


@pytest.fixture(scope="module")
def oracle_files():
    return {lv: [po.encode(lv, px) for _, px in FEATURES] for lv in LEVELS}


def test_walker_consumes_golden_files_exactly():
    """Every golden input at every level: each tile, block and side bit stream ends where its size says, every rANS
    table sums to 2^pb and the context blocks of each tile hold npx - 1 symbols (xw.walk raises otherwise)."""
    seen = set()
    for g, name, e in all_cases(("synthetic", "special", "crops", "corpus"), big=True):
        px = make_case(g, name, e)
        for lv in LEVELS:
            seen |= xw.walk(po.encode(lv, px), lv)
    assert ("v1ctx", "type3") in seen and ("v2ctx", "type4") in seen and ("file", "stored") in seen


def test_feature_set_covers_required(oracle_files):
    seen = set()
    for lv in LEVELS:
        for (name, _), f in zip(FEATURES, oracle_files[lv]):
            seen |= xw.walk(f, lv)
    missing = sorted(REQUIRED - seen, key=str)
    assert not missing, f"the feature set no longer produces {missing}"
    total = sum(px.shape[0] * px.shape[1] for _, px in FEATURES)
    assert 2_100_000 < total < 4_000_000, total   # > 2 MPix: three 1 MPix chunks in the pipelined configuration


def test_unreachable_features(oracle_files):
    """Nothing that is claimed unreachable turns up in the feature set or the golden inputs."""
    feats = set()
    for lv in LEVELS:
        for f in oracle_files[lv]:
            feats |= xw.walk(f, lv)
    for g, name, e in all_cases(("synthetic", "special", "crops", "corpus"), big=False):
        px = make_case(g, name, e)
        for lv in (1, 2):
            feats |= xw.walk(po.encode(lv, px), lv)
    assert not {k for k in feats if k in UNREACHABLE or k[1] in UNREACHABLE}


def _v2_raw_bytes(N, n):
    return 8 + 4 * ((n * xw.bitlen(N - 1) + 31) // 32)


def test_rans_never_wins_below_32_symbols():
    """The bound behind UNREACHABLE["n<32"], from the encoders' own size rules.  A rANS block of n >= 2 symbols over an
    alphabet whose top symbol is N - 1 (at least two used) costs at least its states and its smallest table:
    level 1 (xo_block_v2_encode): 12 header + 16 state bytes + the table in words, raw when that is >= the raw size;
    level 2 (block_v1_encode): 16 state bytes + the table bits, raw when tab_bits + 8 * payload >= nbit * n."""
    for pb in (12, 15):                                   # level 1: contexts (N <= 9, pb 12), alpha (N <= 256, pb 15)
        for N in range(2, 257):
            tab_bits = min(N * pb, N + 2 * pb)            # dense, or sparse with the fewest used symbols
            for n in range(2, 32):
                assert 28 + 4 * ((tab_bits + 31) // 32) >= _v2_raw_bytes(N, n), (pb, N, n)
    for pb, alphabets in ((14, xw.M2_ALPHABET), (15, (256,))):
        for N in alphabets:
            tab_bits = min(N * pb, N + 2 * pb)
            for n in range(2, 32):
                assert tab_bits + 8 * 16 >= xw.bitlen(N - 1) * n, (pb, N, n)


def test_walker_rejects_broken_framing():
    """The walker is not vacuous: a tile size one word off, a flipped table bit, or a truncated file are errors."""
    import struct
    f = bytearray(po.encode(2, synth.rgb(300, 300, 9)))
    bad = bytearray(f)
    struct.pack_into("<I", bad, 8, struct.unpack_from("<I", f, 8)[0] + 4)
    with pytest.raises(xw.WalkError):
        xw.walk(bytes(bad), 2)
    with pytest.raises(xw.WalkError):
        xw.walk(bytes(f[:-4]), 2)
    bad = bytearray(f)
    bad[12 + 3] ^= 0x01            # a bit of the side stream after the first pixel: a table entry
    with pytest.raises(xw.WalkError):
        xw.walk(bytes(bad), 2)
    g = bytearray(po.encode(1, synth.rgb(300, 300, 9)))
    bsz = struct.unpack_from("<I", g, 12)[0]
    q = 12 + bsz                   # first context block; go on to the first rANS block
    while g[q + 3] not in (3, 4):
        q += struct.unpack_from("<I", g, q)[0] & 0xFFFFFF
    w2 =struct.unpack_from("<I", g, q + 8)[0]
    g[q + 8 + 4 * (w2 & 0xFFFFFF) + 3] ^= 0x40
    with pytest.raises(xw.WalkError):
        xw.walk(bytes(g), 1)


# ------------------------------------------------------------------------------------------------------- GPU tests

PAIR = ("k_pd_fill_blocks", "k_dec_rans_pair_v2_ctx", "k_dec_rans_pair_v2_alpha", "k_dec_rans_pair_v1_s8", "k_dec_rans_pair_v1_big",
        "k_dec_walk3<2>")
LAT_TWO = ("k_dec_rans_v2_lat_two", "k_dec_rans_v1_lat_values16_two")
# name -> (environment, kernels that must run, kernels that must not)
CONFIGS = {
    "lat_direct": ({}, ("k_dec_rans_v2_lat", "k_dec_rans_v2_lat_alpha", "k_dec_rans_v1_lat_values16", "k_dec_rans_v1_lat_values256",
                        "k_dec_rans_v1_lat_grey", "k_dec_rans_v1_lat_ctx", "k_dec_rans_v1_lat_ctx_short", "k_dec_walk_smem<0>",
                        "k_dec_unpredict_rows<16>", "k_dec_unpredict", "k_dec_grey_raw", "k_dec_copy", "k_load7"),
                   LAT_TWO + PAIR),
    "lat_two": ({"XPNGB_DIRECT_MAX_TILES": "0", "XPNGB_V2_DIRECT_MAX_TILES": "0"},
                LAT_TWO + ("k_dec_rans_v2_lat_alpha", "k_dec_rans_v1_lat_values256", "k_dec_rans_v1_lat_grey", "k_dec_rans_v1_lat_ctx"),
                ("k_dec_rans_v2_lat", "k_dec_rans_v1_lat_values16", "k_dec_rans_v1_lat_ctx_short") + PAIR),
    "ring": ({"XPNGB_WALK": "ring"}, ("k_dec_walk_ring<1>",), ("k_dec_walk_smem<0>", "k_dec_walk3<2>")),
    "pair_lat16": ({"XPNGB_LAT_MAX_BLOCKS": "0"}, PAIR + ("k_dec_rans_v1_lat_st4",), ("k_dec_rans_pair_v1_s16", "k_dec_rans_v2_lat")),
    "pair_all": ({"XPNGB_LAT_MAX_BLOCKS": "0", "XPNGB_S16_LAT_MAX_TILES": "0"}, PAIR + ("k_dec_rans_pair_v1_s16",),
                 ("k_dec_rans_v1_lat_st4", "k_dec_rans_v2_lat")),
    "pipelined": ({"XPNGB_LAT_MAX_BLOCKS": "0", "XPNGB_PIPE_MIN_MPIX": "1", "XPNGB_CHUNK_MPIX": "1", "XPNGB_PIPE_LANES": "2"},
                  PAIR, ("k_dec_rans_v2_lat",)),
}


def _codec(monkeypatch, env):
    import xpng_b200
    for k, v in env.items():
        monkeypatch.setenv(k, v)      # read by xpngb_create
    return xpng_b200.Codec(0)


def _expected():
    return [po.normalize(px) for _, px in FEATURES]


def _check(got, want, what):
    assert len(got) == len(want)
    for (name, _), g, w in zip(FEATURES * (len(got) // len(FEATURES)), got, want):
        assert g.shape == w.shape and np.array_equal(g, w), (what, name)


def _small_images(n):
    """n images of up to 31 x 28 pixels cut from the feature set, each a tile at levels 1 and 2 (stored and single-colour
    files have none): more than 592 tiles in one call."""
    out, i = [], 0
    while len(out) < n:
        px = FEATURES[i % len(FEATURES)][1]
        h, w = min(px.shape[0], 20 + i % 12), min(px.shape[1], 20 + i % 9)
        y, x = (7 * i) % (px.shape[0] - h + 1), (13 * i) % (px.shape[1] - w + 1)
        crop = np.ascontiguousarray(px[y: y + h, x: x + w])
        if all(xw.walk(po.encode(lv, crop), lv) & {("file", "m1"), ("file", "m2")} for lv in (1, 2)):
            out.append(crop)
        i += 1
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("config", sorted(CONFIGS))
def test_kernel_variant_matrix(monkeypatch, oracle_files, config):
    env, must, must_not = CONFIGS[config]
    cd = _codec(monkeypatch, env)
    want = _expected()
    try:
        calls = [oracle_files[lv] for lv in LEVELS] + [oracle_files[1] + oracle_files[2] + oracle_files[7]]
        for profiled in (True, False):   # profiling serialises launches and bypasses the high-priority stream twin
            cd.profile(profiled)
            for files in calls:
                _check(cd.decode(files), want * (len(files) // len(FEATURES)), (config, profiled))
            if profiled:
                report = cd.profile_report()
                assert not [k for k in must if k not in report], (config, sorted(report))
                assert not [k for k in must_not if k in report], (config, sorted(report))
                if config == "pipelined":   # 2.6 MPix per level in 1 MPix chunks on two lanes: every lane is reused
                    assert report["k_dec_parse_m2"][1] >= 3 and report["k_dec_parse_m1"][1] >= 6, report
        if config == "ring":   # more than 592 tiles: four tiles per CTA, one-warp un-predict
            small = _small_images(640)
            for lv in (1, 2):
                files = [po.encode(lv, px) for px in small]
                for profiled in (True, False):
                    cd.profile(profiled)
                    for g, px in zip(cd.decode(files), small):
                        assert np.array_equal(g, po.normalize(px)), (lv, px.shape, profiled)
                    if profiled:
                        report = cd.profile_report()
                        assert "k_dec_walk_ring<4>" in report and "k_dec_walk_ring<1>" not in report, sorted(report)
                        assert "k_dec_unpredict_rgb" in report or "k_dec_unpredict_rows<1>" in report, sorted(report)
    finally:
        cd.close()


@pytest.mark.gpu
def test_encode_matches_oracle(oracle_files):
    """Encoder choices are part of parity: raw block or rANS, sparse or dense table, grey mode, raw tile, level 7."""
    import xpng_b200
    cd = xpng_b200.Codec(0)
    try:
        imgs = [px for _, px in FEATURES]
        for lv in LEVELS:
            assert cd.encode(lv, imgs) == oracle_files[lv], lv
            for (name, px), want in zip(FEATURES, oracle_files[lv]):
                assert cd.encode(lv, [px])[0] == want, (lv, name)
    finally:
        cd.close()


def _region_cases(oracle_files):
    """Rectangles that start inside a raw tile, a grey raw tile and a single-colour tile (the left tile of each split
    image) and end in the coded tile next to it, at every level."""
    names = [n for n, _ in FEATURES]
    cases = []
    for name, kind in (("split_noise_smooth", ("t2", "raw")), ("split_grey_noise", ("t2", "grey_raw")),
                       ("split_flat_smooth", ("t2", "single"))):
        k = names.index(name)
        assert kind in xw.walk(oracle_files[2][k], 2), name
        for lv in LEVELS:
            for box in ((100, 50, 400, 300), (349, 0, 2, 444), (0, 443, 700, 1), (5, 7, 30, 20)):
                cases.append((oracle_files[lv][k], box))
    assert ("t1", "raw") in xw.walk(oracle_files[1][names.index("split_noise_smooth")], 1)
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("family", ("lat", "pair"))
def test_region_decode_from_special_tiles(monkeypatch, oracle_files, family):
    cd = _codec(monkeypatch, {"XPNGB_LAT_MAX_BLOCKS": "0"} if family == "pair" else {})
    try:
        cases = _region_cases(oracle_files)
        got =cd.decode_region([f for f, _ in cases], [b for _, b in cases])
        for (f, (x, y, w, h)), g in zip(cases, got):
            assert np.array_equal(g, po.decode(f)[y: y + h, x: x + w]), (family, (x, y, w, h))
    finally:
        cd.close()
