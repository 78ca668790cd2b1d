"""LSOP12 and LSOP08 at the edges of their float32 arithmetic, on every decode route.

The coefficients of an LSOP packing are twelve float32 values read from the file (bytes 7..54), so a GVRS file written by
another program may hold any bits there.  The residual streams do not depend on them: rewriting the coefficients (and the
seed, bytes 3..6) of a valid packing gives a packing that still decodes, only to other values.  That puts the prediction
p of a cell exactly where the kernels could go wrong:

- on a half-integer of either sign, and one ulp either side of it (Math.round rounds halves up);
- on -2^21, 2^21 - 1/4 (still inside the fast wavefront's two round-down adds) and on 2^21, -2^21 - 1/4 (outside:
  the tile goes to the general kernels);
- at |p| >= 2^31 (Math.round saturates, the residual add then wraps), on NaN and +-Inf (Math.round(NaN) = 0), on +-0 and
  underflowing products.

Every case is compared with the CPU oracle (oracle.codec_decode_i32) and, on the CPU, the oracle with a second restatement
written here with numpy float32 scalars (lsop12_restated).  The CPU tests also assert that each case reaches the edge it is
named for, so that a change of the base tiles cannot turn an edge case into a plain one.

Which kernels decode a tile cannot be observed; the construction is the evidence (g4_lsop_fast.cu, lsop_fast_geometry and
launch_lsop_decode in g4_lsop.cu):

- fast path (kernels H, T, W): canonical-Huffman packing, tile_cols % 4 == 0 and >= 16, the raster 16-byte aligned.  W and
  pairing follow from tile_cols (ROUTE_SHAPES); `wide` from a raster pitch that is a multiple of 8;
- its exception form (GEN steps): a tile whose interior stream holds residuals outside [-128, 127];
- hand-over to lsop_decode_entropy_kernel + lsop_wavefront_kernel: some p outside [-2^21, 2^21) or NaN, more than 63
  exceptions, a Deflate (type 1) packing, or a packing past the text kernel's staging capacity;
- general aligned (InteriorPackedSink + lsop_wavefront4_kernel): tile_cols 8 or 12;
- general unaligned (InteriorRunSink + lsop_wavefront_kernel): tile_cols % 4 != 0, or a device tile list whose tiles sit
  one int off a 16-byte boundary.
"""
import zlib

import numpy as np
import pytest

from test_gpu_lsop_wave_pairs import SHAPES, _batch, _to_device

INT_MIN, INT_MAX = -(2 ** 31), 2 ** 31 - 1
TWO21 = 2 ** 21

# SHAPES (W 4 / 8 / 16, paired and single) plus single-tile W 8 and W 16 with few rows, general aligned (8, 12 columns) and
# general unaligned (10, 47 columns)
ROUTE_SHAPES = SHAPES + [(40, 200), (24, 288), (30, 8), (21, 12), (26, 10), (33, 47)]
SMALL_SHAPES = [(60, 60), (64, 44), (30, 8), (21, 12), (26, 10), (33, 47)]  # where the numpy restatement runs
TAPS12 = [(0, -1), (-1, -1), (-1, 0), (-1, 1), (-1, 2), (0, -2), (-1, -2), (-2, -2), (-2, -1), (-2, 0), (-2, 1), (-2, 2)]
TAPS08 = [(0, -1), (-1, -1), (-1, 0), (0, -2), (-1, -2), (-2, -2), (-2, -1), (-2, 0)]


# ---- restatement of the reference decoders ------------------------------------------------------------------------------
def _wrap(x):
    """int64 -> the int32 value modulo 2^32."""
    return (np.asarray(x, np.int64) + 2 ** 31) % 2 ** 32 - 2 ** 31


def java_round(p):
    """Math.round(float) (java.lang.Math, JDK >= 7): floor(p + 1/2) in exact arithmetic, NaN -> 0, saturating.  p + 1/2
    is exact in float64 for every float32 p whose magnitude is 2^-30 or more, and below that it cannot cross an integer."""
    x = np.asarray(p, np.float32).astype(np.float64)
    with np.errstate(invalid="ignore"):
        r = np.floor(x + 0.5)
    return np.where(np.isnan(x), 0.0, np.clip(r, INT_MIN, INT_MAX)).astype(np.int64)


def java_f2i(q):
    """(int) q for float32 q: toward zero, NaN -> 0, saturating."""
    x = np.asarray(q, np.float32).astype(np.float64)
    return np.where(np.isnan(x), 0.0, np.clip(np.trunc(np.nan_to_num(x, nan=0.0)), INT_MIN, INT_MAX)).astype(np.int64)


def _stencil(u, v, rows, cols, taps):
    """The float32 stencil of the cells (rows, cols), left to right, one rounding per product and per sum."""
    acc = None
    with np.errstate(all="ignore"):
        for ui, (dr, dc) in zip(u, taps):
            term = ui * v[rows + dr, cols + dc].astype(np.int32).astype(np.float32)
            acc = term if acc is None else acc + term
    return acc


def lsop12_restated(R, C, seed, u, init, interior):
    """LsDecoder12.unpackInitializers + unpackInterior (LsDecoder12.java:204-241, 353-470) over the residual ints.
    Returns (values int32 [R, C], p float32 [R, C], mask): p is the prediction of each interior cell, which `mask` marks."""
    u = [np.float32(x) for x in np.asarray(u, np.float32)]
    init = np.asarray(init, np.int64)
    v = np.zeros((R, C), np.int64)
    k = 0
    v[0, 0] = seed
    for c in range(1, C):
        v[0, c] = _wrap(v[0, c - 1] + init[k]); k += 1
    for r in range(1, R):
        v[r, 0] = _wrap(v[r - 1, 0] + init[k]); k += 1
    for c in range(1, C):
        v[1, c] = _wrap(init[k] + v[1, c - 1] + v[0, c] - v[0, c - 1]); k += 1
    for r in range(2, R):
        v[r, 1] = _wrap(init[k] + v[r, 0] + v[r - 1, 1] - v[r - 1, 0]); k += 1
    tri = init[k:].reshape(R - 2, 2)
    res = np.asarray(interior, np.int64).reshape(R - 2, C - 4)
    p = np.zeros((R, C), np.float32)
    interior_mask = np.zeros((R, C), bool)
    interior_mask[2:, 2:C - 2] = True
    rows_all = np.arange(2, R)
    # cell (r, c) needs (r, c-1), (r, c-2) and rows r-1, r-2 up to column c+2: all on earlier anti-diagonals c + 3r
    for t in range(8, (C - 1) + 3 * (R - 1) + 1):
        cs = t - 3 * rows_all
        sel = (cs >= 2) & (cs < C)
        rs, cs = rows_all[sel], cs[sel]
        inner = cs < C - 2
        ri, ci = rs[inner], cs[inner]
        if ri.size:
            pp = _stencil(u, v, ri, ci, TAPS12)
            p[ri, ci] = pp
            v[ri, ci] = _wrap(java_round(pp) + res[ri - 2, ci - 2])
        for rt, ct in zip(rs[~inner], cs[~inner]):  # Triangle predictor of the last two columns (LsDecoder12.java:459-468)
            v[rt, ct] = _wrap(tri[rt - 2, ct - (C - 2)] + v[rt, ct - 1] + v[rt - 1, ct] - v[rt - 1, ct - 1])
    return v.astype(np.int32), p, interior_mask


def lsop08_restated(R, C, seed, u, init, interior):
    """LsDecoder08.decode (LsDecoder08.java:65-163): the estimate is (int)(p + 0.5f), not Math.round."""
    u = [np.float32(x) for x in np.asarray(u, np.float32)]
    init = np.asarray(init, np.int64)
    v = np.zeros((R, C), np.int64)
    k = 0
    v[0, 0] = seed
    for c in range(1, C):
        v[0, c] = _wrap(v[0, c - 1] + init[k]); k += 1
    prior = seed
    for c in range(C):
        prior = _wrap(prior + init[k]); k += 1
        v[1, c] = prior
    for r in range(2, R):
        v[r, 0] = _wrap(v[r - 1, 0] + init[k]); k += 1
        v[r, 1] = _wrap(v[r, 0] + init[k]); k += 1
    res = np.asarray(interior, np.int64).reshape(R - 2, C - 2)
    p = np.zeros((R, C), np.float32)
    rows_all = np.arange(2, R)
    for t in range(4, (C - 1) + (R - 1) + 1):  # (r, c) needs (r, c-1), (r, c-2) and rows r-1, r-2 up to column c
        cs = t - rows_all
        sel = (cs >= 2) & (cs < C)
        ri, ci = rows_all[sel], cs[sel]
        pp = _stencil(u, v, ri, ci, TAPS08)
        p[ri, ci] = pp
        with np.errstate(all="ignore"):
            q = pp + np.float32(0.5)
        v[ri, ci] = _wrap(java_f2i(q) + res[ri - 2, ci - 2])
    return v.astype(np.int32), p


# ---- packings ---------------------------------------------------------------------------------------------------------
def f32(bits):
    return np.array(bits, np.uint32).view(np.float32)


def coef_bits(taps=None, bits=None, fill=0.0):
    """Twelve coefficients as uint32 bit patterns: `taps` {index: float32 value}, `bits` {index: raw pattern}."""
    u = np.full(12, fill, np.float32).view(np.uint32).copy()
    for i, x in (taps or {}).items():
        u[i] = np.float32(x).view(np.uint32)
    for i, b in (bits or {}).items():
        u[i] = b
    return u


def rewrite(packing, u_bits, seed=None):
    """The packing with its coefficients (and seed) replaced; the streams after the header are untouched."""
    b = bytearray(packing)
    u = np.asarray(u_bits, np.uint32)
    b[7:7 + 4 * u.size] = u.astype("<u4").tobytes()
    if seed is not None:
        b[3:7] = int(_wrap(seed)).to_bytes(4, "little", signed=True)
    return bytes(b)


def seed_of(packing):
    return int.from_bytes(packing[3:7], "little", signed=True)


def lsop12_residuals(oracle, tile):
    """(initializer ints, interior ints) of the tile's packing: the oracle's streams, M32 decoded."""
    _seed, _u, a, b = oracle.lsop12_residual_streams(tile)
    return oracle.m32_decode(a), oracle.m32_decode(b)


def outside_byte(res):
    return int(((res < -128) | (res > 127)).sum())


def terrain(oracle, R, C, k=0):
    """Terrain centred on zero, so that values of both signs occur."""
    t = oracle.terrain_i32(3000 + 37 * k, 500 + 91 * k, R, C).astype(np.int64)
    return (t - int(np.median(t))).astype(np.int32)


def set_residual(oracle, tile, cell, target, tries=8):
    """Moves one interior value until its interior residual is exactly `target` (the refit moves it a little)."""
    R, C = tile.shape
    r, c = cell
    k = (r - 2) * (C - 4) + (c - 2)
    for _ in range(tries):
        res = lsop12_residuals(oracle, tile)[1][k]
        if res == target:
            return True
        v0 = int(tile[r, c]) + int(target - res)
        for j in (1, -1, 2, -2, 3, -3, 0):  # the refit can make the plain step overshoot and oscillate
            tile[r, c] = v0 + j
            if lsop12_residuals(oracle, tile)[1][k] == target:
                return True
    return False


def spiky(oracle, R, C, k=0):
    """Terrain with a few spikes (residuals the text kernel cannot write as a byte) and interior residuals of exactly
    -128 (byte 0, the exception marker), -127, 127 and 128 where the tile has room for them."""
    t = terrain(oracle, R, C, k)
    rng = np.random.default_rng(40 + k)
    for _ in range(max(2, min(8, R * C // 900))):
        r, c = rng.integers(2, R), rng.integers(2, C - 2)
        t[r, c] += int(rng.choice([-1, 1]) * rng.integers(300, 5000))
    if R >= 12 and C >= 16:
        cells = [(R // 4, C // 3), (R // 2, 2 * C // 3), (3 * R // 4, C // 3 + 1), (R - 2, C // 2)]
        k = [(r - 2) * (C - 4) + (c - 2) for r, c in cells]
        for _ in range(20):  # each move refits the tile a little, which may move the residuals set before it
            for cell, target in zip(cells, (-128, -127, 127, 128)):
                set_residual(oracle, t, cell, target)
            if list(lsop12_residuals(oracle, t)[1][k]) == [-128, -127, 127, 128]:
                break
    return t


def repetitive(R, C, k=0):
    """The pattern of test_lsop_deflate_alternative_matches_oracle: LsEncoder12 picks the two zlib streams (type 1)."""
    r, c = np.mgrid[0:R, 0:C]
    return ((r % (3 + k)) * 1000 + (c % (5 + k)) * 37 + (r // 16) * 5 + (r * c) % (2 + k) - 1000).astype(np.int32)


# coefficient sets: name -> (bits, base tile kind, level) -- `level` is where the seed moves the values (None: unchanged)
SETS = {
    "half+": (coef_bits({0: 0.5}), "terrain", None),
    "half-": (coef_bits({0: -0.5}), "terrain", None),
    "half+ulp": (coef_bits(bits={0: 0x3F000001}), "terrain", None),   # 0.5 + 2^-24
    "half-ulp": (coef_bits(bits={0: 0x3EFFFFFF}), "terrain", None),   # 0.5 - 2^-25
    # p = 1.125 a - 0.375 b + 0.25 c is a multiple of 1/8; near 1.5 * 2^20 the float32 spacing is 1/8, near 3 * 2^20 it
    # is 1/4 (outside the fast range).  The taps sum to 1, so the level set by the seed holds across the tile.
    "eighths": (coef_bits({0: 1.125, 5: -0.375, 2: 0.25}), "terrain", 3 * 2 ** 19),
    "quarters": (coef_bits({0: 1.125, 5: -0.375, 2: 0.25}), "terrain", 3 * 2 ** 20),
    "range-lo-in": (coef_bits({0: 1.0}), "terrain", ("min", -TWO21)),                      # p = -2^21: fast
    "range-hi-in": (coef_bits(bits={0: 0x3F7FFFFE}), "terrain", ("max", TWO21)),         # 1 - 2^-23: p = 2^21 - 1/4
    "range-hi-out": (coef_bits({0: 1.0}), "terrain", ("max", TWO21)),                     # p = 2^21: handed over
    "range-lo-out": (coef_bits(bits={0: 0x3F800001}), "terrain", ("min", -TWO21)),        # 1 + 2^-23: p = -2^21 - 1/4
    "saturate": (coef_bits({0: 1024.0}), "terrain", 2 ** 22),
    "saturate-": (coef_bits({0: 1024.0}), "terrain", -(2 ** 22)),
    "nan": (coef_bits(bits={0: 0x7FC00000}), "terrain", None),
    "nan-payload": (coef_bits({0: 0.5}, bits={3: 0x7F8A5A5A, 7: 0xFFC0BEEF}), "terrain", None),
    "+inf": (coef_bits(bits={0: 0x7F800000}), "terrain", None),
    "-inf": (coef_bits(bits={2: 0xFF800000}), "terrain", None),
    "0*inf": (coef_bits({0: 0.5}, bits={9: 0x7F800000}), "zeros", None),
    "subnormal": (coef_bits({0: 0.5}, bits={1: 0x00000001, 2: 0x807FFFFF, 3: 0x00400000}), "terrain", None),
    "zeros": (coef_bits(), "negative", None),
    "-0": (coef_bits(fill=-0.0), "positive", None),
}


def _base_tile(oracle, kind, R, C, spikes):
    if kind == "zeros":  # mostly zeros: products 0 * Inf
        rng = np.random.default_rng(R * 1000 + C)
        t = np.where(rng.random((R, C)) < 0.5, 0, rng.integers(-3, 4, (R, C))).astype(np.int32)
        return t
    t = spiky(oracle, R, C) if spikes else terrain(oracle, R, C)
    if kind == "negative":
        return (t - int(t.max()) - 5).astype(np.int32)
    if kind == "positive":
        return (t - int(t.min()) + 5).astype(np.int32)
    return t


def _leveled(oracle, packing, R, C, u_bits, level):
    """The packing with coefficients u_bits and its seed moved so that the values sit at `level`.  ("min"/"max", x):
    the smallest / largest value that feeds the u0 tap, v[r][c-1] for interior cells, lands on x exactly -- decoded with
    u0 = 1, whose values move with the seed one for one (|v| < 2^24); 1 +- 2^-23 decodes to the same values below 2^22."""
    if level is None:
        return rewrite(packing, u_bits)
    if isinstance(level, tuple):
        v = oracle.codec_decode_i32(oracle.CODEC_LSOP12, R, C, rewrite(packing, coef_bits({0: 1.0})))
        feed = v[2:, 1:C - 3].astype(np.int64)
        delta = level[1] - (feed.min() if level[0] == "min" else feed.max())
    else:
        delta = level - seed_of(packing)
    return rewrite(packing, u_bits, seed_of(packing) + delta)


class Case:
    def __init__(self, name, R, C, packing, init, interior, base):
        self.name, self.R, self.C, self.packing = name, R, C, packing
        self.init, self.interior, self.base = init, interior, base


_CACHE = {}


def crafted_cases(oracle, R, C):
    """Every coefficient set on the plain and the spiky base tile (canonical-Huffman form), and a few on the Deflate
    form where LsEncoder12 picks it.  Cached per shape."""
    key = (R, C)
    if key in _CACHE:
        return _CACHE[key]
    cases = []
    bases = {}
    for name, (u_bits, kind, level) in SETS.items():
        for spikes in (False, True):
            if kind != "terrain" and spikes:
                continue
            bk = (kind, spikes)
            if bk not in bases:
                tile = _base_tile(oracle, kind, R, C, spikes)
                p = oracle.lsop12_encode(0, tile, deflate=False)
                assert p is not None and p[1] & 0x0F == 2, (R, C, bk)
                bases[bk] = (tile, p, lsop12_residuals(oracle, tile))
            tile, p, (init, interior) = bases[bk]
            cases.append(Case(name + ("/spiky" if spikes else ""), R, C, _leveled(oracle, p, R, C, u_bits, level), init, interior, tile))
    rep = repetitive(R, C)
    p = oracle.lsop12_encode(0, rep, deflate=True)
    if p is not None and p[1] & 0x0F == 1:
        init, interior = lsop12_residuals(oracle, rep)
        for name in ("half+", "range-hi-out", "range-lo-in", "saturate", "nan", "0*inf"):
            u_bits, _kind, level = SETS[name]
            cases.append(Case(name + "/deflate", R, C, _leveled(oracle, p, R, C, u_bits, level), init, interior, rep))
    _CACHE[key] = cases
    return cases


def oracle_decode(oracle, case):
    return oracle.codec_decode_i32(oracle.CODEC_LSOP12, case.R, case.C, case.packing)


def restated(case):
    return lsop12_restated(case.R, case.C, seed_of(case.packing), f32(np.frombuffer(case.packing[7:55], "<u4")),
                           case.init, case.interior)


# ---- what each case must reach (CPU) ------------------------------------------------------------------------------------
def _is_half(p):
    x = p.astype(np.float64)
    with np.errstate(invalid="ignore"):
        return np.isfinite(x) & (x - np.floor(x) == 0.5)


def _next_to_half(p):
    """p one float32 ulp above / below a half-integer."""
    x = p.astype(np.float64)
    fin = np.isfinite(x)
    up = np.nextafter(p, np.float32(-np.inf)).astype(np.float64)
    dn = np.nextafter(p, np.float32(np.inf)).astype(np.float64)
    with np.errstate(invalid="ignore"):
        above = fin & (up - np.floor(up) == 0.5) & ~_is_half(p)
        below = fin & (dn - np.floor(dn) == 0.5) & ~_is_half(p)
    return above, below


def edge_counts(case, p, mask):
    """Counts of the edges this case's predictions p reach, over its interior cells."""
    q = p[mask]
    x = q.astype(np.float64)
    half = _is_half(q)
    above, below = _next_to_half(q)
    with np.errstate(invalid="ignore"):
        fast = bool(np.all((x >= -TWO21) & (x < TWO21)))
        n = {
            "half>0": int((half & (x > 0)).sum()), "half<0": int((half & (x < 0)).sum()),
            "half+1ulp": int(above.sum()), "half-1ulp": int(below.sum()),
            "half@1/8": int((half & (np.abs(x) >= 2 ** 20) & (np.abs(x) < TWO21)).sum()),
            "half@1/4": int((half & (np.abs(x) >= TWO21) & (np.abs(x) < 2 ** 22)).sum()),
            "p=-2^21": int((x == -TWO21).sum()), "p=2^21-1/4": int((x == TWO21 - 0.25).sum()),
            "p=2^21": int((x == TWO21).sum()), "p=-2^21-1/4": int((x == -TWO21 - 0.25).sum()),
            "p>=2^31": int((x >= 2.0 ** 31).sum()), "p<=-2^31": int((x <= -(2.0 ** 31)).sum()),
            "nan": int(np.isnan(x).sum()), "+inf": int((x == np.inf).sum()), "-inf": int((x == -np.inf).sum()),
            "-0": int(((x == 0) & np.signbit(q)).sum()), "+0": int(((x == 0) & ~np.signbit(q)).sum()),
        }
    n["fast"] = fast
    return n


# the edges each set must reach, and whether its tile stays inside the fast range (None: not asserted)
EXPECT = {
    "half+": (["half>0", "half<0"], True),
    "half-": (["half>0", "half<0"], True),
    "half+ulp": (["half+1ulp"], True),
    "half-ulp": (["half-1ulp"], True),
    "eighths": (["half@1/8"], True),
    "quarters": (["half@1/4"], False),
    "range-lo-in": (["p=-2^21"], True),
    "range-hi-in": (["p=2^21-1/4"], True),
    "range-hi-out": (["p=2^21"], False),
    "range-lo-out": (["p=-2^21-1/4"], False),
    "saturate": (["p>=2^31", "p<=-2^31"], False),
    "saturate-": (["p>=2^31", "p<=-2^31"], False),
    "nan": (["nan"], False),
    "nan-payload": (["nan"], False),
    "+inf": (["+inf", "-inf"], False),
    "-inf": (["+inf", "-inf"], False),
    "0*inf": (["nan", "+inf"], False),
    "subnormal": (["half>0", "half<0"], True),
    "zeros": (["-0"], True),
    "-0": (["-0"], True),
}


def _subnormal_products(case):
    """Products u_i * z_i of the subnormal set that are subnormal, over the interior values of the base tile."""
    u = f32(np.frombuffer(case.packing[7:55], "<u4"))
    z = case.base[2:, 2:case.C - 2].astype(np.float32)
    with np.errstate(all="ignore"):
        prods = [u[i] * z for i in (1, 2, 3)]
    return sum(int(((np.abs(x) < np.float32(2.0 ** -126)) & (x != 0)).sum()) for x in prods)


@pytest.mark.parametrize("shape", SMALL_SHAPES)
def test_crafted_cases_reach_their_edges_and_the_oracle_agrees(oracle, shape):
    """CPU: the oracle decodes every crafted packing to the numpy restatement's values, and every case reaches the edges
    its set is named for (EXPECT), on the plain and on the spiky base tile."""
    R, C = shape
    cases = crafted_cases(oracle, R, C)
    for case in cases:
        want, p, mask = restated(case)
        got = oracle_decode(oracle, case)
        assert np.array_equal(got, want), "%s %s: oracle != restatement" % (shape, case.name)
        n = edge_counts(case, p, mask)
        if case.name.endswith("/deflate"):  # there for the route (type 1 is always handed over), not for an edge
            continue
        set_name = case.name.split("/")[0]
        kinds, fast = EXPECT[set_name]
        for kind in kinds:
            assert n[kind] > 0, "%s %s: no cell with %s (%s)" % (shape, case.name, kind, n)
        if fast is not None:
            assert n["fast"] == fast, "%s %s: fast range %s, expected %s" % (shape, case.name, n["fast"], fast)
        if set_name == "subnormal":
            assert _subnormal_products(case) > 0, case.name
    if C % 4 == 0 and C >= 16:
        assert any(c.name.endswith("/deflate") for c in cases), "%s: no Deflate-form case" % (shape,)
    for c in cases:
        if c.name.endswith("/spiky") and R >= 12 and C >= 16:
            res = c.interior
            assert outside_byte(res) > 0 and outside_byte(res) <= 63, (shape, outside_byte(res))
            assert {-128, -127, 127, 128} <= set(res.tolist()), shape
            break


def test_restated_rounding_matches_the_oracle(oracle):
    """CPU: java_round / java_f2i above against the oracle's Math.round on the awkward values."""
    vals = [0.5, -0.5, 1.5, -1.5, 2.5, -2.5, 0.49999997, -0.49999997, 2.0 ** 21 - 0.5, -(2.0 ** 21) - 0.5, 2.0 ** 23 + 1,
            2.0 ** 31, -(2.0 ** 31), 3e9, -3e9, np.inf, -np.inf, np.nan, 1e-45, -1e-45, -0.0, 8388607.5]
    for x in vals:
        assert java_round(np.float32(x)) == oracle.java_round(float(np.float32(x))), x


# ---- 5b: the rounding identity of the fast wavefront (CPU) ---------------------------------------------------------------
def _fadd_rd(a, b):
    """__fadd_rd on float32 arrays: the float64 sum is exact here; round it to float32, one ulp down if that went up."""
    s = a.astype(np.float64) + b.astype(np.float64)
    r = s.astype(np.float32)
    return np.where(r.astype(np.float64) > s, np.nextafter(r, np.float32(-np.inf)), r)


def test_two_round_down_adds_equal_math_round_near_every_half_and_the_range_ends():
    """CPU: t1 = RD(p + 1.5*2^22), t2 = RD(t1 + 1.5*2^22 + 1/2) gives 1.5*2^23 + Math.round(p) for every float32 within
    two ulps of every k + 1/2, k in [-2^21, 2^21], and of +-2^21 -- and t1's exponent flags exactly the p outside
    [-2^21, 2^21) (the kernel's range check, g4_lsop_fast.cu lsop3_wave_kernel).  About 21 M values."""
    magic_half, magic_half_up = np.float32(6291456.0), np.float32(6291456.5)
    offs = np.array([-2, -1, 0, 1, 2], np.int32)
    edges = np.array([TWO21, -TWO21], np.float32).view(np.int32)
    step = 1 << 20
    checked = 0
    for k0 in range(-TWO21, TWO21 + 1, step):
        ks = np.arange(k0, min(k0 + step, TWO21 + 1), dtype=np.float64)
        base = (ks + 0.5).astype(np.float32).view(np.int32)
        if k0 == -TWO21:
            base = np.concatenate([base, edges])
        p = (base[:, None] + offs[None, :]).ravel().view(np.float32)
        t1 = _fadd_rd(p, magic_half)
        t2 = _fadd_rd(t1, magic_half_up)
        fast = (t2.astype(np.float64) - 12582912.0).astype(np.int64)
        flagged = ((t1.view(np.uint32) ^ np.uint32(0x4A800000)) & np.uint32(0xFF800000)) != 0
        x = p.astype(np.float64)
        inside = (x >= -TWO21) & (x < TWO21)
        assert np.array_equal(flagged, ~inside), p[flagged != ~inside][:8]
        want = java_round(p)
        bad = inside & (fast != want)
        assert not bad.any(), (p[bad][:8], fast[bad][:8], want[bad][:8])
        checked += int(inside.sum())
    assert checked > 20_000_000


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def g4():
    import gridfour_b200

    return gridfour_b200


def _master(g4):
    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("LSOP12", g4.LsEncoder12, g4.LsDecoder12)
    return g4.CodecMaster(spec)


def _diff(got, want):
    d = np.argwhere(np.asarray(got) != np.asarray(want))
    return "%d cells differ, first at %s: %s != %s" % (len(d), tuple(d[0]), got[tuple(d[0])], want[tuple(d[0])]) if len(d) else ""


def _decode_band(g4, master, payloads, R, C, extra, device):
    """The payloads as one band row of tiles inside a raster `extra` columns wider (grid_pitch = n C + extra)."""
    n = len(payloads)
    band = master._band((R, n * C), np.int32, R, C)
    band.grid_pitch = n * C + extra
    batch = _batch(g4, payloads, band)
    out = np.full((R, n * C + extra), -7, np.int32)
    if device:
        import torch

        o = torch.from_numpy(out).cuda()
        master.decodeTiles(_to_device(g4, batch), out=o)
        raster, st = o.cpu().numpy(), master.lastStatus.cpu().numpy()
    else:
        raster, st = master.decodeTiles(batch, out=out), np.asarray(master.lastStatus)
    assert np.all(raster[:, n * C:] == -7), "columns past the band were written"
    return [raster[:, t * C:(t + 1) * C] for t in range(n)], st


def _decode_list(g4, master, payloads, R, C, pitch, shift, device):
    """decodeTileList: tile t at offset t * (R + 1) * pitch + shift, rows `pitch` apart."""
    import torch

    n = len(payloads)
    b = _batch(g4, payloads, None)
    refs = [(t * (R + 1) * pitch + shift, pitch) for t in range(n)]
    out = np.full(n * (R + 1) * pitch + shift + 8, -7, np.int32)
    if device:
        dev = torch.from_numpy(out).cuda()
        master.decodeTileList(torch.from_numpy(b.arena).cuda(), torch.from_numpy(b.offsets.astype(np.int64)).cuda(),
                              torch.from_numpy(b.lens.astype(np.int32)).cuda(), dev, refs, R, C)
        out = dev.cpu().numpy()
    else:
        master.decodeTileList(b.arena, b.offsets, b.lens, out, refs, R, C)
    return [out[o:o + R * p].reshape(R, p)[:, :C] for o, p in refs]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ROUTE_SHAPES)
def test_crafted_coefficients_decode_like_the_oracle_on_every_route(g4, oracle, shape):
    """Every crafted case through LsDecoder12.decode, decodeTiles from host and device in rasters of pitch 8 and 4 mod 8
    past the band, and decodeTileList from host and device with 16-byte aligned, 4-int and 1-int offset tiles."""
    R, C = shape
    cases = crafted_cases(oracle, R, C)
    wants = [oracle_decode(oracle, c) for c in cases]
    payloads = [c.packing for c in cases]
    dec = g4.LsDecoder12()
    for c, w in zip(cases, wants):
        got = dec.decode(R, C, c.packing)
        assert np.array_equal(got, w), "%s %s single: %s" % (shape, c.name, _diff(got, w))
    master = _master(g4)
    for device in (False, True):
        for extra in (8, 4):
            tiles, st = _decode_band(g4, master, payloads, R, C, extra, device)
            assert not np.any(st), (shape, device, extra, st)
            for c, w, got in zip(cases, wants, tiles):
                assert np.array_equal(got, w), "%s %s band device=%s +%d: %s" % (shape, c.name, device, extra, _diff(got, w))
        for pitch, shift in ((C + 8 - C % 8, 8), (C + 4 + (4 - C % 4) % 4, 4), (C + 3, 1)):
            for c, w, got in zip(cases, wants, _decode_list(g4, master, payloads, R, C, pitch, shift, device)):
                assert np.array_equal(got, w), "%s %s list device=%s pitch %d +%d: %s" % (shape, c.name, device, pitch, shift,
                                                                                           _diff(got, w))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [s for s in ROUTE_SHAPES if s[1] % 4 == 0 and s[1] >= 16])
def test_both_sides_of_the_fast_range_in_one_warp(g4, oracle, shape):
    """Bands of exactly two tiles (one pair where tile_cols gives two tiles per warp): one tile whose predictions stay in
    [-2^21, 2^21) next to one that reaches 2^21 or -2^21 - 1/4, in both orders, plain and with exceptions."""
    R, C = shape
    by_name = {c.name: c for c in crafted_cases(oracle, R, C)}
    master = _master(g4)
    for sfx in ("", "/spiky"):
        for a, b in (("range-lo-in", "range-hi-out"), ("range-hi-out", "range-lo-in"), ("range-hi-in", "range-lo-out"),
                     ("range-lo-out", "range-hi-in"), ("eighths", "quarters")):
            ca, cb = by_name[a + sfx], by_name[b + sfx]
            for device in (False, True):
                tiles, st = _decode_band(g4, master, [ca.packing, cb.packing], R, C, 0, device)
                for c, got in zip((ca, cb), tiles):
                    w = oracle_decode(oracle, c)
                    assert np.array_equal(got, w), "%s %s next to %s: %s" % (shape, c.name, (cb if c is ca else ca).name, _diff(got, w))


# ---- 3: route boundaries that are counts ----------------------------------------------------------------------------------
EXC_CAP = 63  # kExcCap of g4_lsop_fast.cu: a tile with more exceptions leaves the fast path
EXC_SHAPES = [(180, 240), (60, 60)]


def exceptions_tile(oracle, R, C, target):
    """Terrain with spikes added one at a time until exactly `target` interior residuals are no byte (counted in the
    oracle's interior stream)."""
    t = terrain(oracle, R, C, 7)
    rng = np.random.default_rng(1000 + target + R)
    n = outside_byte(lsop12_residuals(oracle, t)[1])
    for _ in range(3000):
        if n == target:
            return t
        cand = t.copy()
        r, c = rng.integers(2, R), rng.integers(2, C - 2)
        cand[r, c] += int(rng.choice([-1, 1]) * rng.integers(140, 400))
        m = outside_byte(lsop12_residuals(oracle, cand)[1])
        if m <= target:
            t, n = cand, m
    raise AssertionError("no tile with %d exceptions" % target)


def fast_stage_limit(R, C):
    """Largest canonical packing the fast text kernel stages (text_stage_words; kernel H defers len + 96 > 4 words)."""
    w = (R * C * 5 // 8 + 3) // 4 + 128
    w = max(w, 512)
    return 4 * ((w + 255) & ~255) - 96


def general_stage_limit(R, C):
    """Largest canonical packing lsop_decode_text_kernel stages (stageWords of launch_lsop_decode)."""
    w = min(max((R * C * 5 // 8 + 3) // 4, 7168), 49152)
    return 4 * ((w + 255) & ~255)


def sized_tiles(oracle, R, C, limit):
    """Two noise tiles whose canonical packings are at most `limit` bytes and one more cell of wider noise past it: the
    number of wide cells is bisected."""
    rng = np.random.default_rng(R * C)
    narrow = rng.integers(-12, 13, (R, C))
    wide = rng.integers(-200, 201, (R, C))
    order = rng.permutation(R * C)

    def tile(k):
        t = narrow.copy().ravel()
        t[order[:k]] = wide.ravel()[order[:k]]
        return t.reshape(R, C).astype(np.int32)

    def size(k):
        return len(oracle.lsop12_encode(0, tile(k), deflate=False))

    lo, hi = 0, R * C
    assert size(lo) <= limit < size(hi), (size(lo), limit, size(hi))
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if size(mid) <= limit:
            lo = mid
        else:
            hi = mid
    return tile(lo), tile(hi)


STAGE_CASES = [(180, 240, "fast"), (180, 238, "general")]


def _stage_tiles(oracle, R, C, kind):
    limit = fast_stage_limit(R, C) if kind == "fast" else general_stage_limit(R, C)
    return limit, sized_tiles(oracle, R, C, limit)


def test_counted_boundaries_sit_where_they_are_claimed(oracle):
    """CPU: the tiles of the exception-list and staging tests are on the two sides of their counts, and the spiky base
    tiles of the fast shapes keep their exceptions within the list."""
    for R, C in EXC_SHAPES:
        for target in (EXC_CAP, EXC_CAP + 1):
            assert outside_byte(lsop12_residuals(oracle, exceptions_tile(oracle, R, C, target))[1]) == target
    for R, C, kind in STAGE_CASES:
        limit, (a, b) = _stage_tiles(oracle, R, C, kind)
        la, lb = len(oracle.lsop12_encode(0, a, deflate=False)), len(oracle.lsop12_encode(0, b, deflate=False))
        assert la <= limit < lb and lb - la < 16, (R, C, kind, la, limit, lb)
    for R, C in ROUTE_SHAPES:
        if C % 4 == 0 and C >= 16:
            res = lsop12_residuals(oracle, spiky(oracle, R, C))[1]
            assert 0 < outside_byte(res) <= EXC_CAP, (R, C, outside_byte(res))
            assert {-128, -127, 127, 128} <= set(res.tolist()), (R, C)


def _decode_everywhere(g4, oracle, packings, R, C, what):
    """Single-tile decode, and a band of all packings from host and device, against the oracle."""
    wants = [oracle.codec_decode_i32(oracle.CODEC_LSOP12, R, C, p) for p in packings]
    for k, (p, w) in enumerate(zip(packings, wants)):
        got = g4.LsDecoder12().decode(R, C, p)
        assert np.array_equal(got, w), "%s %d single: %s" % (what, k, _diff(got, w))
    master = _master(g4)
    for device in (False, True):
        tiles, st = _decode_band(g4, master, packings, R, C, 0, device)
        assert not np.any(st), (what, device, st)
        for k, (got, w) in enumerate(zip(tiles, wants)):
            assert np.array_equal(got, w), "%s %d band device=%s: %s" % (what, k, device, _diff(got, w))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", EXC_SHAPES)
def test_exception_list_full_and_one_past_it(g4, oracle, shape):
    """Interior streams with exactly 63 (the list's capacity: fast path, GEN steps) and 64 (handed over) residuals that are
    no byte, as they are and with the coefficients rewritten to u0 = 0.5; the two share a warp in the band."""
    R, C = shape
    packings = []
    for target in (EXC_CAP, EXC_CAP + 1):
        p = oracle.lsop12_encode(0, exceptions_tile(oracle, R, C, target), deflate=False)
        packings += [p, rewrite(p, coef_bits({0: 0.5}))]
    _decode_everywhere(g4, oracle, [packings[0], packings[2]], R, C, "exceptions")
    _decode_everywhere(g4, oracle, [packings[1], packings[3]], R, C, "exceptions, u0 = 0.5")


@pytest.mark.gpu
@pytest.mark.parametrize("case", STAGE_CASES)
def test_packings_at_the_text_kernels_staging_capacity(g4, oracle, case):
    """Canonical packings of at most / just past what the fast text kernel (180 x 240) or the general text kernel
    (180 x 238, unaligned) stages; past it the general entropy kernel decodes the tile."""
    R, C, kind = case
    _limit, (a, b) = _stage_tiles(oracle, R, C, kind)
    pa, pb = oracle.lsop12_encode(0, a, deflate=False), oracle.lsop12_encode(0, b, deflate=False)
    _decode_everywhere(g4, oracle, [pa, pb], R, C, kind)
    _decode_everywhere(g4, oracle, [rewrite(pa, coef_bits({0: 0.5})), rewrite(pb, coef_bits({0: -0.5}))], R, C, kind + " rewritten")


# ---- 4: the encoder's summation order -------------------------------------------------------------------------------------
TH_R, TH_C = 34, 68  # nInterior = 32 * 64 = 2^11, so max|z| = 2^21 puts nInterior * max|z|^2 exactly on 2^53


def threshold_tiles(oracle):
    """name -> tile: the largest magnitude one below, on and one above 2^21 (in a corner: max|z| is over all cells),
    and tiles of mixed magnitudes or far from zero, far above, where the two summation orders round differently."""
    base = terrain(oracle, TH_R, TH_C, 3)
    out = {}
    for name, m in (("below", TWO21 - 1), ("at", TWO21), ("above", TWO21 + 1), ("at-", -TWO21)):
        t = base.copy()
        t[0, 0] = m
        out[name] = t
    rng = np.random.default_rng(53)
    for k in range(4):
        big = rng.integers(-(2 ** 30), 2 ** 30, (TH_R, TH_C))
        t = np.where(rng.random((TH_R, TH_C)) < 0.3, big, base + rng.integers(-50, 50, (TH_R, TH_C)))
        out["mixed%d" % k] = t.astype(np.int32)
    # samples far from zero with small differences: the normal equations are ill-conditioned, so a change in the last
    # bit of a sum moves the float32 coefficients
    for e in (22, 24, 26):
        for amp in (50, 5000):
            out["offset%d/%d" % (e, amp)] = (2 ** e + base + rng.integers(-amp, amp, (TH_R, TH_C))).astype(np.int32)
    return out


def _moment_terms(tile):
    """Per interior cell, in the reference's cell order, z_0 ... z_12 (LsOptimalPredictor12.computeCoefficients)."""
    R, C = tile.shape
    taps = [(0, 0)] + TAPS12
    v = tile.astype(np.float64)
    return np.stack([v[2 + dr:R + dr, 2 + dc:C - 2 + dc].ravel() for dr, dc in taps])


def _sequential(x):
    s = 0.0
    for a in x:
        s += a
    return s


def _partitioned(x):
    """lsop_encode_kernel's order: 64 lanes take every 64th cell, each half-warp set of 32 lanes reduces by xor shuffles,
    then the two halves are added."""
    lanes = [_sequential(x[l::64]) for l in range(64)]
    halves = []
    for g in (0, 1):
        v = np.array(lanes[32 * g:32 * g + 32])
        for d in (16, 8, 4, 2, 1):
            v = v + v[np.arange(32) ^ d]
        halves.append(v[0])
    return halves[0] + halves[1]


def test_threshold_tiles_sit_on_their_side_of_2_53(oracle):
    """CPU: nInterior * max|z|^2 against 2^53 for each tile, and for the tiles above it at least one moment whose
    partitioned and sequential float64 sums differ."""
    tiles = threshold_tiles(oracle)
    n_int = (TH_R - 2) * (TH_C - 4)
    for name, t in tiles.items():
        prod = n_int * int(np.abs(t.astype(np.int64)).max()) ** 2
        side = "below" if prod < 2 ** 53 else "at" if prod == 2 ** 53 else "above"
        assert side == {"below": "below", "at": "at", "above": "above", "at-": "at"}.get(name, "above"), (name, side)
    for name, t in tiles.items():
        if name in ("below", "at", "above", "at-"):
            continue
        z = _moment_terms(t)
        differ = 0
        for i in range(13):
            for j in range(i, 13):
                x = z[i] * z[j]
                differ += _sequential(x) != _partitioned(x)
        assert differ > 0, name


@pytest.mark.gpu
def test_encoder_packings_at_the_summation_threshold(g4, oracle):
    """LsEncoder12 on the GPU equals the oracle byte for byte (coefficients, both streams, option bits) on every side of
    nInterior * max|z|^2 = 2^53, for both options on and off, per tile and batched."""
    tiles = threshold_tiles(oracle)
    packed = 0
    for name, t in tiles.items():
        for deflate in (False, True):
            for checksum in (False, True):
                want = oracle.lsop12_encode(0, t, deflate=deflate, checksum=checksum)
                e = g4.LsEncoder12()
                e.setDeflateEnabled(deflate)
                e.setValueChecksumEnabled(checksum)
                got = e.encode(0, TH_R, TH_C, t)
                assert got == want, "%s deflate=%s checksum=%s: %s" % (name, deflate, checksum,
                                                                        None if got is None or want is None else _diff(np.frombuffer(got, np.uint8), np.frombuffer(want, np.uint8)))
                packed += want is not None
    assert packed >= 20
    names = list(tiles)
    grid = np.concatenate([tiles[n] for n in names], axis=1)
    batch = _master(g4).encodeTiles(grid, TH_R, TH_C)
    for k, n in enumerate(names):  # the CodecMaster rule: LSOP12, or raw where that is shorter
        assert batch.payload(k) == oracle.master_encode_i32([oracle.CODEC_LSOP12], tiles[n]), n


# ---- 5a: LSOP08, whose estimate truncates p + 0.5f ------------------------------------------------------------------------
LSOP08_SHAPES = [(40, 50), (61, 77), (90, 120)]
LSOP08_SETS = {"-0.7": coef_bits({0: -0.7}), "0.3/-0.55": coef_bits({0: 0.3, 2: -0.55}), "half-": coef_bits({0: -0.5})}


def lsop08_streams(oracle, packing):
    """(seed, initializer ints, interior ints) of an LSOP08 packing (revised header, LsDecoder08.java:65-110)."""
    typ = packing[1] & 0x0F
    n_init = int.from_bytes(packing[39:43], "little")
    n_int = int.from_bytes(packing[43:47], "little")
    body = packing[47:]
    if typ == 0:
        n_int &= 0xFFFFFF  # LsEncoder08.java:122 clears the top byte of the second count
        a, pos = oracle.huffman_decode_at(body, n_init, 0)
        b, _ = oracle.huffman_decode_at(body, n_int, pos)
    else:
        d = zlib.decompressobj()
        a = d.decompress(body)
        b = zlib.decompress(d.unused_data)
    return seed_of(packing), oracle.m32_decode(a), oracle.m32_decode(b)


def lsop08_cases(oracle):
    out = []
    for R, C in LSOP08_SHAPES:
        p = oracle.lsop08_encode(0, terrain(oracle, R, C, 5))
        seed, init, interior = lsop08_streams(oracle, p)
        for name, u in LSOP08_SETS.items():
            out.append(("%dx%d %s" % (R, C, name), R, C, rewrite(p, u[:8]), seed, u[:8], init, interior, p[1] & 0x0F))
    return out


def test_lsop08_restatement_and_where_truncation_is_not_rounding(oracle):
    """CPU: the oracle's LSOP08 decode of the rewritten packings equals the restatement, and the cases hold negative,
    non-half p where (int)(p + 0.5f) differs from Math.round (and from round-to-nearest-even)."""
    types = set()
    for name, R, C, p, seed, u, init, interior, typ in lsop08_cases(oracle):
        types.add(typ)
        want, pp = lsop08_restated(R, C, seed, f32(u), init, interior)
        assert np.array_equal(oracle.lsop08_decode(R, C, p), want), name
        q = pp[2:, 2:]
        with np.errstate(all="ignore"):
            trunc = java_f2i(q + np.float32(0.5))
        x = q.astype(np.float64)
        assert ((x < 0) & ~_is_half(q) & (trunc != java_round(q)) & (trunc != np.rint(x))).sum() > 0, name
    assert types == {0, 1} or len(types) == 1  # whichever body the encoder picked; both are decoded the same way


@pytest.mark.gpu
def test_lsop08_rewritten_coefficients_decode_like_the_reference(g4, oracle):
    """LsDecoder08 on the GPU, per tile and batched, against the oracle and the restatement."""
    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("LSOP08", g4.LsEncoder08, g4.LsDecoder08)
    master = g4.CodecMaster(spec)
    by_shape = {}
    for name, R, C, p, seed, u, init, interior, _typ in lsop08_cases(oracle):
        want = oracle.lsop08_decode(R, C, p)
        assert np.array_equal(want, lsop08_restated(R, C, seed, f32(u), init, interior)[0]), name
        got = g4.LsDecoder08().decode(R, C, p)
        assert np.array_equal(got, want), "%s: %s" % (name, _diff(got, want))
        by_shape.setdefault((R, C), []).append((p, want))
    for (R, C), items in by_shape.items():
        for device in (False, True):
            tiles, st = _decode_band(g4, master, [p for p, _w in items], R, C, 0, device)
            assert not np.any(st), st
            for (p, w), got in zip(items, tiles):
                assert np.array_equal(got, w), "%dx%d band device=%s: %s" % (R, C, device, _diff(got, w))
