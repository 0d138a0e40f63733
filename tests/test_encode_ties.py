"""Every size decision of the encoder driven to its exact tie, and the GPU's files compared with the CPU oracle there.

The encoder writes the reference's bytes only if each of its size comparisons goes the same way as the reference's,
including when the two sides are equal: coded or raw tile, coded or stored file, rANS or raw block, sparse or dense
table, the predictor and grey-candidate picks, and the donor of the frequency "steal".  Ordinary images almost never
produce those ties, so a `<` turned `<=` would pass every other test.  Here small deterministic image families with one
integer knob are searched against the oracle's decision log (pyoracle.encode_traced) for inputs where a comparison is
exactly tied, next to an input one knob step away where it goes the other way.  REQUIRED_TIES names what must be
found; UNREACHABLE_TIES lists the ties no input can produce, with the arithmetic checked.  An oracle built with each
comparison flipped must write a different file for some input found.  The GPU tests encode the inputs found and compare
every byte with the oracle, then decode them.
"""
import numpy as np
import pytest

from oracle import pyoracle as po
import xpng_walk as xw

TWO_SIDED = (po.D_T1_TILE, po.D_FILE, po.D_T2_TILE, po.D_GREY_PLANE, po.D_V2_BLOCK, po.D_V2_TABLE, po.D_V1_BLOCK,
             po.D_V1_TABLE)
PICKS = (po.D_PRED, po.D_GREY_PICK)
NL_DIFF = (0, -1, 1, 2, 4, 8, 16, 32, 64)   # a left difference whose zig-zag has bit length nl = 0..8

# --------------------------------------------------------------------------------------------------------- images


def noise_prefix(h, w, c, seed, grey=False):
    """k -> an h x w tile whose first k pixels (row-major) are noise and the rest flat: the coded size grows with k
    past the raw size."""
    rng = np.random.default_rng(seed)
    noise = rng.integers(0, 256, (h * w, c), dtype=np.uint8)
    if grey:
        noise[:, 1] = noise[:, 2] = noise[:, 0]
    flat = np.full((h * w, c), 77, np.uint8)
    if c == 4:
        noise[:, 3] = rng.integers(1, 255, h * w)   # translucent, never 0: the image stays RGBA and nothing is zeroed
        flat[:, 3] = 128

    def make(k):
        px = flat.copy()
        px[:k] = noise[:k]
        return px.reshape(h, w, c)
    return make


def grey_band(seed):
    """k -> a 24 x 24 grey tile v = f(x + y) + g(x - y), f a random walk and g a staircase that rises at most 1 over
    two diagonals, so that every left neighbour is the upper one or 1 below it: the up and avg2 candidates are the same
    residual plane (left and grad3 are others).  k is added to the pixel above the last: it changes the last pixel's
    up and avg2 residuals differently, so a tie of candidates 1 and 2 at one k breaks at the next."""
    rng = np.random.default_rng(seed)
    n = 24
    f = 128 + np.cumsum(rng.choice([-2, -1, 0, 1, 2, 3], 2 * n))
    steps = rng.random(4 * n) < 0.4
    g = np.zeros(4 * n, np.int64)
    for i in range(2, 4 * n):
        g[i] = g[i - 1] + int(steps[i] and g[i - 1] == g[i - 2])
    y, x = np.mgrid[0:n, 0:n]
    base = f[x + y] + g[x - y + 2 * n]

    def make(k):
        v = base.copy()
        v[n - 2, n - 1] += k
        return np.repeat((v % 256).astype(np.uint8)[..., None], 3, axis=2)
    return make


def two_tiles(seed, c=3, flat_first=False):
    """k -> two tiles of noise (RGB: one row of 295705 pixels, tiles 147853 and 147852 wide; RGBA: 4 rows of 73927,
    tiles 36964 and 36963 wide, xo_tile_grid), the last k columns of the second tile flat: its coded size crosses its
    raw size near here.  With a noise first tile (raw) the file decision sees the sum of both; with a flat first tile
    the file stays coded, so a tie of the second tile shows in the file."""
    rng = np.random.default_rng(seed)
    h, w, w0 = (1, 295705, 147853) if c == 3 else (4, 73927, 36964)
    noise = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
    if c == 4:
        noise[..., 3] = rng.integers(1, 255, (h, w))
    if flat_first:
        noise[:, :w0] = 60

    def make(k):
        px = noise.copy()
        px[:, w - k:] = 9
        return px
    return make


def predictor_tile(c):
    """k -> a 16 x 16 tile whose 16 predictor samples (pixel (3 + 4i, 3 + 4j) and its left, upper and upper-left
    neighbours, xo_select_predictor) are set one by one.  A type-T sample costs (4, 3, 4, 3), a type-W sample (1, 1, 0,
    0); samples 0 .. k-1 are W.  k = 0 ties predictors 1 and 3 at 48 above 64; k = 1 picks 3."""
    def make(k):
        px = np.full((16, 16, c), 100, np.uint8)
        if c == 4:
            px[..., 3] = 200
        for s in range(16):
            y, x = 3 + 4 * (s // 4), 3 + 4 * (s % 4)
            if s < k:   # W: upper-left 2 above, pixel 1 below: avg2 residual -1 in every channel, grad3 residual 0
                px[y - 1, x - 1, :3] = 102
                px[y, x, :3] = 99
            else:       # T: flat neighbours, pixel +(4, 1, 4)
                px[y, x, :3] = (104, 101, 104)
        return px
    return make


def alpha_image(sym, h, w):
    """Flat RGB over an alpha plane whose level-1 alpha stream (zig-zag left differences, column 0 from above) is sym."""
    s = np.asarray(sym, np.int64)
    assert len(s) == h * w - 1
    d = np.zeros(h * w, np.int64)
    d[1:] = (s >> 1) ^ -(s & 1)
    d = d.reshape(h, w)
    d[0, 0] = 128
    a = (np.cumsum(d[:, 0])[:, None] + np.cumsum(np.concatenate([np.zeros((h, 1), np.int64), d[:, 1:]], axis=1),
                                                 axis=1)) % 256
    assert a.min() > 0 and a.max() < 255, "alpha must stay translucent and non-zero"
    px = np.empty((h, w, 4), np.uint8)
    px[..., :3] = (40, 90, 200)
    px[..., 3] = a
    return px


def alpha_table(k):
    """k = used symbols of a 15-symbol alpha alphabet (top symbol 14 always used): 15 + 15 k against 15 * 15 table
    bits, a tie at k = 14 (dense) next to k = 13 (sparse)."""
    seq = np.zeros(8 * 64 - 1, np.int64)
    used = list(range(1, k - 1)) + [14]
    for i, s in enumerate(used):
        seq[10 + 20 * i] = s
        seq[20 + 20 * i] = s - 1 if s % 2 else s   # undo the step so that alpha stays near 128
    return alpha_image(seq, 8, 64)


def alpha_noise(seed):
    """k -> an 8 x 64 RGBA tile, flat RGB, whose first k alpha differences are in -4 .. 3: the alpha block's rANS
    size crosses its raw size."""
    rng = np.random.default_rng(seed)
    sym = rng.integers(0, 8, 8 * 64 - 1)

    def make(k):
        s = np.zeros(8 * 64 - 1, np.int64)
        s[:k] = sym[:k]
        return alpha_image(s, 8, 64)
    return make


def scattered(counts, n, rng):
    """n symbols: symbol s + 1 counts[s] times at random places, the rest 0."""
    seq = np.zeros(n, np.int64)
    pos = rng.permutation(n)[: sum(counts)]
    k = 0
    for s, c in enumerate(counts, 1):
        seq[pos[k: k + c]] = s
        k += c
    return seq


def steal_counts(k, nsym):
    """Counts of symbols 1 .. nsym - 1 for knob k: symbols of count 1 round to width 0 when the block holds about twice
    2^pb symbols, symbols of count 4 are width-2 donors.  The top symbol is used."""
    rng = np.random.default_rng(k)
    c = [int(v) for v in rng.choice([0, 1, 1, 4, 4], nsym - 1)]
    c[-1] = max(c[-1], 1)
    return c, rng


def alpha_steal(k):
    """4 x 16384 RGBA (one tile, 65535 alpha symbols, pb 15): the steal of the alpha block."""
    return alpha_image(alpha_image_symbols(k), 4, 16384)


def row_image(nls):
    """One row whose residuals (left differences, channel 0 only) have bit lengths nls: the context stream of each
    previous nl is set symbol by symbol, at level 1 (no predictor below 4 rows) and level 2 alike."""
    d = np.array([0] + [NL_DIFF[v] for v in nls], np.int64)
    px = np.empty((1, len(d), 3), np.uint8)
    px[0, :, 0] = (100 + np.cumsum(d)) % 256
    px[0, :, 1:] = (30, 170)
    return px


def alpha_steal_counts(k):
    """The symbol counts of alpha_steal(k)'s alpha block."""
    return np.bincount(alpha_image_symbols(k), minlength=15).tolist()


def alpha_image_symbols(k):
    c, rng = steal_counts(k, 15)
    return scattered(c, 4 * 16384 - 1, rng)


def row_steal_nls(k, width):
    c, _ = steal_counts(100 + k, 9)
    nls = []
    for s, n in enumerate(c, 1):
        nls += [s, 0] * n
    return nls + [0] * (width - 1 - len(nls))


def row_steal(width):
    """k -> one row of `width` pixels whose context-0 block holds about `width` symbols with the counts of
    steal_counts(k, 9) after it (8300: pb 12 at level 1, over 4096; 33000: pb 14 at level 2, over 16384)."""
    return lambda k: row_image(row_steal_nls(k, width))


def row_steal_counts(width):
    """k -> the symbol counts of row_steal(width)(k)'s context-0 block: the nl of each pixel that follows an nl of 0."""
    def counts(k):
        nls = row_steal_nls(k, width)
        return np.bincount([b for a, b in zip([0] + nls[:-1], nls) if a == 0], minlength=9).tolist()
    return counts


def row_used(k):
    """One row whose context-0 block uses all 9 symbols (k = 0) or all but symbol k: both sides of the sparse/dense
    boundary of a 9-symbol table (used 8 and 9), at level 1 (pb 12) and level 2 (pb 14)."""
    nls = []
    for s in range(1, 9):
        if s != k:
            nls += [s, 0] * 4
    return row_image(nls + [0] * 200)


def row_values(seed):
    """k -> one row of k pixels after the first with nl = 1, most of them -1 in channel 0 only: the level-2 value
    stream of nl = 1 (8 symbols, 3 bits raw) crosses from raw to rANS."""
    rng = np.random.default_rng(seed)
    v = np.where(rng.random(400) < 0.6, 4, rng.integers(1, 8, 400))
    d = -np.stack([(v >> 2) & 1, (v >> 1) & 1, v & 1], axis=1)

    def make(k):
        px = np.empty((1, k + 1, 3), np.int64)
        px[0, 0] = (100, 50, 200)
        px[0, 1:] = px[0, 0] + np.cumsum(d[:k], axis=0)
        return (px % 256).astype(np.uint8)
    return make


# name -> (levels, knobs, k -> image)
FAMILIES = {}
for _s in range(4):
    FAMILIES[f"prefix_rgb{_s}"] = ((1, 2), range(257), noise_prefix(16, 16, 3, _s))
    FAMILIES[f"prefix_rgba{_s}"] = ((1, 2), range(257), noise_prefix(16, 16, 4, _s))
    FAMILIES[f"prefix_grey{_s}"] = ((2,), range(257), noise_prefix(16, 16, 3, _s, grey=True))
    FAMILIES[f"alpha_noise{_s}"] = ((1,), range(511), alpha_noise(_s))
FAMILIES["two_tiles"] = ((1, 2), range(1160, 1270), two_tiles(0))
for _s in range(4):
    FAMILIES[f"flat_and_noise{_s}"] = ((1, 2), range(1160, 1270), two_tiles(_s, flat_first=True))
    FAMILIES[f"flat_and_noise_rgba{_s}"] = ((1,), range(300, 340), two_tiles(_s, 4, flat_first=True))
for _s in (14, 29, 44):
    FAMILIES[f"grey_band{_s}"] = ((2,), range(8), grey_band(_s))
FAMILIES["row_used"] = ((1, 2), range(3), row_used)
FAMILIES["pred_rgb"] = ((1, 2), range(3), predictor_tile(3))
FAMILIES["pred_rgba"] = ((1, 2), range(3), predictor_tile(4))
FAMILIES["alpha_table"] = ((1, 2), range(12, 16), alpha_table)
FAMILIES["alpha_steal"] = ((1,), range(24), alpha_steal)
FAMILIES["row_steal_pb12"] = ((1,), range(8), row_steal(8300))
FAMILIES["row_steal_pb14"] = ((2,), range(8), row_steal(33000))
# steal families -> k -> the symbol counts of the block that steals
STEAL_BLOCKS = {"alpha_steal": alpha_steal_counts, "row_steal_pb12": row_steal_counts(8300),
                "row_steal_pb14": row_steal_counts(33000)}
for _s in range(4):
    FAMILIES[f"row_values{_s}"] = ((2,), range(120, 220), row_values(_s))

# ------------------------------------------------------------------------------------------------ what must be hit

# (decision, level, channels, pb or stream class) -> families searched for it.  pb: the block's probability bits
# (level 1: 12 contexts, 15 alpha; level 2: 14).
_PREFIX = lambda kind: tuple(f"prefix_{kind}{s}" for s in range(4))
REQUIRED_TIES = {
    # a tile tie shows only in a file that stays coded, hence a flat tile beside the tied one
    ("t1_tile", 1, 3, None): tuple(f"flat_and_noise{s}" for s in range(4)),
    ("t1_tile", 1, 4, None): tuple(f"flat_and_noise_rgba{s}" for s in range(4)),
    ("file", 1, 3, None): _PREFIX("rgb"),
    ("file", 1, 4, None): _PREFIX("rgba"),
    ("file", 2, 3, None): _PREFIX("rgb"),
    ("file_two_tiles", 1, 3, None): ("two_tiles",),
    ("file_two_tiles", 2, 3, None): ("two_tiles",),
    ("t2_tile", 2, 3, None): tuple(f"flat_and_noise{s}" for s in range(4)),
    ("grey_plane", 2, 3, None): _PREFIX("grey"),
    ("grey_pick", 2, 3, None): tuple(f"grey_band{s}" for s in (14, 29, 44)),
    ("pred", 1, 3, None): ("pred_rgb",),
    ("pred", 2, 3, None): ("pred_rgb",),
    ("pred", 1, 4, None): ("pred_rgba",),
    ("v2_block", 1, 3, 12): _PREFIX("rgb"),
    ("v2_block", 1, 4, 12): _PREFIX("rgba"),
    ("v2_block", 1, 4, 15): tuple(f"alpha_noise{s}" for s in range(4)),
    ("v2_table", 1, 4, 15): ("alpha_table",),
    ("v2_table", 2, 4, 15): ("alpha_table",),
    ("v1_block", 2, 3, 14): tuple(f"row_values{s}" for s in range(4)),
    ("steal", 1, 4, 15): ("alpha_steal",),
    ("steal", 1, 3, 12): ("row_steal_pb12",),
    ("steal", 2, 3, 14): ("row_steal_pb14",),
}
# The steal's cases, each in a block that stays rANS (so that the table is in the file): several donors of the same
# smallest width with the first taken, the donor before and after the starved symbol, two starved symbols in a block.
STEAL_CASES = ("tied_donors", "donor_before", "donor_after", "two_starved")

# Ties no input can produce, with the arithmetic (test_unreachable_ties checks each).  For the two table forms the
# neighbouring `used` counts on both sides of the boundary are required instead (NEIGHBOUR_USED).
UNREACHABLE_TIES = {
    ("v2_table", 12): "sparse N + 12 used = dense 12 N needs 12 used = 11 N, so 12 | N; the level-1 context alphabets "
                      "have N <= 9",
    ("v1_table", 14): "N + 14 used = 14 N needs 14 | N; the level-2 alphabets are 9, 8, 64, 8, 16, 32, 64, 128, 256",
    ("v1_table", 15): "N + 15 used = 15 N with N = 256 (grey) needs 15 | 256",
    ("v1_block_ctx", 14): "a level-2 context block (N = 9, 4 bits raw) compares 126 or 9 + 14 used table bits plus "
                          "128 + 32 words of states and words with 4 n: the left side is 2 mod 4 or odd",
}
# (decision, pb, N) -> the two `used` counts either side of the sparse/dense boundary, both required.
NEIGHBOUR_USED = {
    ("v2_table", 12, 9): (8, 9),
    ("v1_table", 14, 9): (8, 9),
}

# ------------------------------------------------------------------------------------------------------ the search


def _key(r):
    return int(r["kind"]), int(r["tile"]), int(r["stream"])


class Run:
    """One family at one level: the files and logs of every knob value."""

    def __init__(self, name, lv):
        self.name, self.lv = name, lv
        _, knobs, self.make = FAMILIES[name]
        self.knobs = list(knobs)
        self.files, self.logs = [], []
        for k in self.knobs:   # the images are made again when needed: a family can be a few hundred MB of them
            px = self.make(k)
            f, log = po.encode_traced(lv, px)
            self.files.append(f)
            self.logs.append(log)
        self.c = px.shape[2]

    def image(self, i):
        return self.make(self.knobs[i])

    def records(self, i, kind):
        log = self.logs[i]
        return log[log["kind"] == kind]

    def first(self, i, key):
        for r in self.logs[i]:
            if _key(r) == key:
                return r
        return None


def _tie(r):
    k = int(r["kind"])
    v = [int(x) for x in r["v"]]
    if k in TWO_SIDED:
        return v[0] == v[1]
    if k in PICKS:
        m = min(v)
        tied = [i for i in range(4) if v[i] == m]
        return m > 0 and len(tied) >= 2 and 0 not in tied
    return False


def _pb_of(run, r):
    """Probability bits of the block a record belongs to: level 2 RGB (not grey) 14, level 1 contexts 12, alpha 15."""
    if run.lv == 2 and run.c == 3:
        return 14
    return 15 if int(r["stream"]) == 9 else 12


_KIND = {"t1_tile": po.D_T1_TILE, "file": po.D_FILE, "file_two_tiles": po.D_FILE, "t2_tile": po.D_T2_TILE,
         "grey_plane": po.D_GREY_PLANE, "grey_pick": po.D_GREY_PICK, "pred": po.D_PRED, "v2_block": po.D_V2_BLOCK,
         "v2_table": po.D_V2_TABLE, "v1_block": po.D_V1_BLOCK, "steal": po.D_STEAL}


def find_tie(run, what, pb):
    """(knob index of the tie, knob index of its neighbour) for decision `what`, or None."""
    kind = _KIND[what]
    for i in range(len(run.knobs)):
        for r in run.records(i, kind):
            if not _tie(r) or (pb is not None and _pb_of(run, r) != pb):
                continue
            if what == "file_two_tiles" and int(r["v"][2]) != 2:
                continue
            if not _visible(run.logs[i], r):
                continue
            for j in (i - 1, i + 1):
                if 0 <= j < len(run.knobs):
                    o = run.first(j, _key(r))
                    if o is not None and int(o["outcome"]) != int(r["outcome"]):
                        return i, j
    return None


def _visible(log, r):
    """Whether decision r can show in the file: the file is coded, the tile is coded (a stored file holds no tile, a
    raw tile no block), a block is in the tile (grey: the picked candidate's) and a table belongs to a rANS block."""
    kind, tile, stream = _key(r)
    if kind == po.D_FILE:
        return True
    f = log[log["kind"] == po.D_FILE]
    if len(f) != 1 or int(f[0]["outcome"]) != 1:
        return False
    if kind in (po.D_T1_TILE, po.D_T2_TILE, po.D_GREY_PLANE):
        return True
    L = log[log["tile"] == tile]
    t = L[np.isin(L["kind"], [po.D_T1_TILE, po.D_T2_TILE, po.D_GREY_PLANE])]
    if len(t) != 1 or int(t[0]["outcome"]) != 1:
        return False
    grey = L[L["kind"] == po.D_GREY_PICK]
    if kind in (po.D_PRED, po.D_GREY_PICK):
        return True
    if len(grey) and int(grey[0]["outcome"]) != stream:
        return False
    if kind in (po.D_V2_TABLE, po.D_V1_TABLE, po.D_STEAL):
        b = L[np.isin(L["kind"], [po.D_V2_BLOCK, po.D_V1_BLOCK]) & (L["stream"] == stream)]
        return len(b) == 1 and int(b[0]["outcome"]) == 1
    return True


def normalise(F, pb, last=False):
    """normalise_freqs of xpng_oracle.c: (final widths, [(starved symbol, donor)]).  last=True takes the last of the
    donors of equal smallest width instead of the first, which is what a `<=` in the donor search would do."""
    N, n = len(F), sum(F)
    cum = [0]
    for f in F:
        cum.append(cum[-1] + f)
    cum = [0] + [(c << pb) // n for c in cum[1:]]
    steals = []
    for i in range(N):
        if F[i] and cum[i + 1] == cum[i]:
            w = [cum[j + 1] - cum[j] for j in range(N)]
            cand = [j for j in range(N) if w[j] > 1]
            best = min(w[j] for j in cand)
            tied = [j for j in cand if w[j] == best]
            donor = tied[-1] if last else tied[0]
            if donor < i:
                for j in range(donor + 1, i + 1):
                    cum[j] -= 1
            else:
                for j in range(i + 1, donor + 1):
                    cum[j] += 1
            steals.append((i, donor))
    return [cum[j + 1] - cum[j] for j in range(N)], steals


def steal_cases(run, pb):
    """STEAL_CASES -> knob index where it happens in a block that stays rANS in a coded tile.  Tied donors count only
    where taking the last of them instead of the first leaves a different table (a later steal can undo the choice)."""
    found = {}
    counts = STEAL_BLOCKS[run.name]
    for i in range(len(run.knobs)):
        log = run.logs[i]
        rec = [r for r in log[log["kind"] == po.D_STEAL] if _pb_of(run, r) == pb and _visible(log, r)]
        if not rec:
            continue
        stream = {int(r["stream"]) for r in rec}
        assert len(stream) == 1, stream
        F = counts(run.knobs[i])
        widths, steals = normalise(F, pb)
        assert steals == [(int(r["v"][0]), int(r["outcome"])) for r in rec], (run.name, i)   # normalise is the oracle's
        if len(rec) >= 2:
            found.setdefault("two_starved", i)
        for r in rec:
            starved, donor, ties = int(r["v"][0]), int(r["outcome"]), int(r["v"][2])
            found.setdefault("donor_before" if donor < starved else "donor_after", i)
            if ties >= 2 and normalise(F, pb, last=True)[0] != widths:
                found.setdefault("tied_donors", i)
    return found


_runs = {}


def run(name, lv):
    if (name, lv) not in _runs:
        _runs[(name, lv)] = Run(name, lv)
    return _runs[(name, lv)]


def search():
    """REQUIRED_TIES entry -> (family, knob index of the tie, knob index of the neighbour); steals -> their cases."""
    hits = {}
    for (what, lv, c, pb), fams in REQUIRED_TIES.items():
        for name in fams:
            if lv not in FAMILIES[name][0]:
                continue
            R = run(name, lv)
            if what == "steal":
                cases = steal_cases(R, pb)
                if all(k in cases for k in STEAL_CASES):
                    hits[(what, lv, c, pb)] = (name, cases)
                    break
                continue
            t = find_tie(R, what, pb)
            if t:
                hits[(what, lv, c, pb)] = (name,) + t
                break
    return hits


@pytest.fixture(scope="module")
def ties():
    return search()


def tie_images(hits):
    """Every input that a hit names (the tie and its neighbour, every steal case), once, with the level it is for."""
    out, seen = [], set()
    for key, h in sorted(hits.items(), key=str):
        lv = key[1]
        idx = sorted(set(h[1].values())) if key[0] == "steal" else [h[1], h[2]]
        for i in idx:
            if (h[0], i) not in seen:
                seen.add((h[0], i))
                out.append((f"{h[0]}[{FAMILIES[h[0]][1][i]}]", run(h[0], lv).image(i)))
    for k in FAMILIES["row_used"][1]:   # NEIGHBOUR_USED: both sides of the boundary where no tie can be
        out.append((f"row_used[{k}]", row_used(k)))
    return out

# -------------------------------------------------------------------------------------------------------- CPU tests


def test_required_ties_are_hit(ties):
    missing = sorted(set(REQUIRED_TIES) - set(ties), key=str)
    assert not missing, f"no tie with a neighbour on the other side found for {missing}"
    for key, h in ties.items():
        if key[0] == "steal":
            continue
        name, i, j = h
        R = run(name, key[1])
        assert R.c == key[2] and abs(i - j) == 1, (key, h)


def test_tie_outcomes_follow_the_reference(ties):
    """At a tie the reference keeps the raw tile, the stored file, the raw block, the dense table and the lowest
    predictor or grey candidate; the log says so for every hit."""
    for key, h in ties.items():
        if key[0] == "steal":
            continue
        name, i, _ = h
        for r in run(name, key[1]).records(i, _KIND[key[0]]):
            if not _tie(r):
                continue
            if int(r["kind"]) in PICKS:
                v = [int(x) for x in r["v"]]
                assert int(r["outcome"]) == v.index(min(v)), (key, r)
            else:
                assert int(r["outcome"]) == 0, (key, r)


def test_unreachable_ties():
    """The arithmetic behind UNREACHABLE_TIES, over every table size and block length the encoders can meet."""
    for N in range(2, 10):                                 # level-1 contexts, pb 12
        for used in range(2, N + 1):
            assert N + 12 * used != 12 * N, (N, used)
    for N in set(xw.M2_ALPHABET):                          # level 2, pb 14
        for used in range(2, N + 1):
            assert N + 14 * used != 14 * N, (N, used)
    for used in range(2, 257):                             # grey, pb 15
        assert 256 + 15 * used != 15 * 256, used
    for nw in range(0, 1 << 12):                           # level-2 contexts: N = 9, 4 bits a symbol
        for tab in [9 * 14] + [9 + 14 * u for u in range(2, 9)]:
            assert (tab + 128 + 32 * nw) % 4 != 0, (tab, nw)
    # the other tables do tie: 15 + 15 * 14 = 15 * 15 (alpha, pb 15, top symbol 14 with 14 used)
    assert 15 + 15 * 14 == 15 * 15


def test_neighbour_used_counts():
    """For the ties that cannot occur, both sides of the sparse/dense boundary next to it are still met, each in a rANS
    block of a coded tile (so that the table form is in the file the GPU tests compare)."""
    seen = set()
    kinds = {po.D_V2_TABLE: "v2_table", po.D_V1_TABLE: "v1_table"}
    for name in ("row_used",):
        for lv in FAMILIES[name][0]:
            R = run(name, lv)
            for log in R.logs:
                for r in log[np.isin(log["kind"], list(kinds))]:
                    pb = 12 if int(r["kind"]) == po.D_V2_TABLE else 14
                    if int(r["kind"]) == po.D_V2_TABLE and int(r["stream"]) == 9 or not _visible(log, r):
                        continue
                    seen.add((kinds[int(r["kind"])], pb, int(r["v"][3]), int(r["v"][2]), int(r["outcome"])))
    for (what, pb, N), (lo, hi) in NEIGHBOUR_USED.items():
        assert (what, pb, N, lo, 1) in seen, (what, pb, N, lo, "sparse")
        assert (what, pb, N, hi, 0) in seen, (what, pb, N, hi, "dense")


def test_steal_cases(ties):
    for key in [k for k in REQUIRED_TIES if k[0] == "steal"]:
        name, cases = ties[key]
        assert set(STEAL_CASES) <= set(cases), (key, cases)


def test_trace_changes_no_output(ties):
    """Encoding with the decision log on writes the same bytes as with it off."""
    from xpng_b200 import synth
    imgs = [px for _, px in tie_images(ties)] + [synth.rgb(300, 300, 1), synth.rgba(64, 80, 2), synth.noise(40, 50, 3)]
    for px in imgs:
        for lv in (1, 2, 7):
            f, log = po.encode_traced(lv, px)
            assert f == po.encode(lv, px)
    assert po.encode_traced(1, synth.rgb(300, 300, 1))[1].size > 0


# Each size comparison of the oracle with its tie sent the other way, as a one-token edit of xpng_oracle.c.  The
# kernels restate the same lines (enc_back.cuh, enc_m2.cuh, enc_rans_lat.cuh, common.cuh pick_predictor).
FLIPS = {
    "t1_tile": ("if (coded < raw)", "if (coded <= raw)"),
    "file": ("if (total >= s)", "if (total > s)"),
    "grey_pick": ("if (bsz[i] + rsz[i] < bsz[best] + rsz[best])", "if (bsz[i] + rsz[i] <= bsz[best] + rsz[best])"),
    "grey_plane": ("if (bsz[best] + rsz[best] >= npx) {", "if (bsz[best] + rsz[best] > npx) {"),
    "t2_tile": ("if (bsz + rsz >= npx * 3)", "if (bsz + rsz > npx * 3)"),
    "v2_table": ("int sparse = (N + used * (unsigned)pb) < N * (unsigned)pb;",
                 "int sparse = (N + used * (unsigned)pb) <= N * (unsigned)pb;"),
    "v1_table": ("int sparse = tab_bits < N * (uint32_t)pb;", "int sparse = tab_bits <= N * (uint32_t)pb;"),
    "v2_block": ("if (csz >= rawsz)", "if (csz > rawsz)"),
    "v1_block": ("if (tab_bits + 8 * payload >= (uint64_t)nbit * n)", "if (tab_bits + 8 * payload > (uint64_t)nbit * n)"),
    "pred": ("if (cost[k] < cost[m]) m = k;", "if (cost[k] <= cost[m]) m = k;"),
    "steal": ("wdt > 1 && wdt < best", "wdt > 1 && wdt <= best"),
}


def test_flipped_oracle_comparisons_change_the_tie_set(ties, tmp_path):
    """The tie set bites: an oracle built with any one comparison flipped writes a different file for at least one
    tie input, except the v1 table flip, which no input can tell apart (UNREACHABLE_TIES)."""
    import os
    import subprocess
    imgs = tie_images(ties)
    want = {lv: [po.encode(lv, px) for _, px in imgs] for lv in (1, 2)}
    src = open(os.path.join(os.path.dirname(po.__file__), "xpng_oracle.c")).read()
    saved = po._lib, po._LIB
    try:
        for name, (a, b) in FLIPS.items():
            assert src.count(a) == 1, name
            c, so = tmp_path / f"{name}.c", tmp_path / f"{name}.so"
            c.write_text(src.replace(a, b))
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-I" + os.path.dirname(po.__file__), "-o", str(so), str(c)],
                           check=True)
            po._lib, po._LIB = None, str(so)
            changed = [(lv, n) for lv in (1, 2) for (n, px), w in zip(imgs, want[lv]) if po.encode(lv, px) != w]
            assert bool(changed) == (name != "v1_table"), (name, changed)
    finally:
        po._lib, po._LIB = saved


def _check_log_against_file(f, log, lv):
    """The log agrees with the file: every non-empty, non-run block of every coded tile has one rANS/raw record whose
    outcome is the block's kind, every table record its table form, and the tile and file records their kinds."""
    tiles = []
    xw.walk(f, lv, tiles)
    mode = f[3]
    frec = log[log["kind"] == po.D_FILE]
    if frec.size:
        assert int(frec[0]["outcome"]) == (mode != 7)
    if mode == 7:
        assert not tiles
        return 0
    checked = 0
    for t, (m, kinds) in enumerate(tiles):
        L = log[log["tile"] == t]
        tile_rec = L[np.isin(L["kind"], [po.D_T1_TILE, po.D_T2_TILE, po.D_GREY_PLANE])]
        if m in (0, 0x28):          # raw tile or raw grey plane
            assert int(tile_rec[-1]["outcome"]) == 0, (t, m)
            continue
        if m == 255:
            assert tile_rec.size == 0
            continue
        assert int(tile_rec[-1]["outcome"]) == 1, (t, m)
        blocks = L[np.isin(L["kind"], [po.D_V2_BLOCK, po.D_V1_BLOCK])]
        tables = L[np.isin(L["kind"], [po.D_V2_TABLE, po.D_V1_TABLE])]
        if m >> 4 == 2:             # grey: only the picked candidate is in the file
            pick = int(L[L["kind"] == po.D_GREY_PICK][0]["outcome"])
            assert m & 3 == pick
            blocks, tables = blocks[blocks["stream"] == pick], tables[tables["stream"] == pick]
        coded = [(s, k) for s, k in enumerate(kinds) if k in (2, 3, 4)]
        assert len(coded) == blocks.size == tables.size, (t, coded, blocks)
        for (s, k), b, tb in zip(coded, blocks, tables):
            assert int(b["stream"]) == s or m >> 4 == 2, (t, s, b)
            assert int(b["outcome"]) == (k != 2), (t, s, k, b)
            if k != 2:
                assert int(tb["outcome"]) == (k == 4), (t, s, k, tb)
            checked += 1
    return checked


def test_log_agrees_with_the_file(ties):
    """Non-vacuity: the records counted and compared here are the blocks and tiles the walker reads in the file."""
    n = 0
    for _, px in tie_images(ties):
        for lv in (1, 2):
            f, log = po.encode_traced(lv, px)
            n += _check_log_against_file(f, log, lv)
    from test_block_coverage import FEATURES
    for _, px in FEATURES[:12]:
        for lv in (1, 2):
            f, log = po.encode_traced(lv, px)
            n += _check_log_against_file(f, log, lv)
    assert n > 100, n

# -------------------------------------------------------------------------------------------------------- GPU tests


@pytest.fixture(scope="module")
def tie_set(ties):
    imgs = tie_images(ties)
    return imgs, {lv: [po.encode(lv, px) for _, px in imgs] for lv in (1, 2)}


@pytest.mark.gpu
def test_encode_ties_match_oracle(tie_set):
    """Each tie input alone, all in one batch, and the batch reversed (k_enc_order's sorted work lists put blocks of
    different images side by side): every file equals the oracle's byte for byte."""
    import xpng_b200
    imgs, want = tie_set
    cd = xpng_b200.Codec(0)
    try:
        for lv in (1, 2):
            for (name, px), w in zip(imgs, want[lv]):
                assert cd.encode(lv, [px])[0] == w, (lv, name, "alone")
            got = cd.encode(lv, [px for _, px in imgs])
            for (name, _), g, w in zip(imgs, got, want[lv]):
                assert g == w, (lv, name, "batch")
            got = cd.encode(lv, [px for _, px in imgs][::-1])[::-1]
            for (name, _), g, w in zip(imgs, got, want[lv]):
                assert g == w, (lv, name, "reversed batch")
    finally:
        cd.close()


@pytest.mark.gpu
@pytest.mark.parametrize("family", ("lat", "pair"))
def test_decode_ties(monkeypatch, tie_set, family):
    import xpng_b200
    if family == "pair":
        monkeypatch.setenv("XPNGB_LAT_MAX_BLOCKS", "0")
    imgs, want = tie_set
    cd = xpng_b200.Codec(0)
    try:
        for lv in (1, 2):
            for (name, px), g in zip(imgs, cd.decode(want[lv])):
                assert np.array_equal(g, po.normalize(px)), (family, lv, name)
    finally:
        cd.close()
