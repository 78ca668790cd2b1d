"""-m gpu: the LSOP12 strip wavefront with two tiles per warp.

Tiles whose columns fit 16 strips (60 to 256 columns in the terrain configs) are decoded two per warp, one per 16-lane
half, in the order of the LSOP tile list.  That order comes from an atomic counter, so a test cannot choose which tiles
share a warp; a band that holds exactly two LSOP12 tiles, however, always decodes them as one pair.  Every decode here
must give the input back wherever the oracle decodes the tile, whatever its partner is: a tile with exceptions, one the
text kernel or the wavefront hands to the general kernels, one that fails, or no partner at all."""
import itertools

import numpy as np
import pytest

from gridfour_b200._lib import G4_ERR_FORMAT, G4_OK

pytestmark = pytest.mark.gpu

KINDS = ["plain", "few", "many", "range", "spike", "malformed"]


@pytest.fixture(scope="module")
def g4():
    import gridfour_b200

    return gridfour_b200


def _master(g4, names=("LSOP12",)):
    std = {"GvrsHuffman": (g4.CodecHuffman, g4.CodecHuffman), "GvrsDeflate": (g4.CodecDeflate, g4.CodecDeflate),
           "LSOP12": (g4.LsEncoder12, g4.LsDecoder12)}
    spec = g4.CodecSpecification(default=False)
    for n in names:
        spec.addCompressionCodec(n, *std[n])
    return g4.CodecMaster(spec)


def _kind_tile(oracle, kind, k, tr=180, tc=240):
    """The tile kinds of test_lsop_fast_path_exception_and_range_tiles_in_a_band: residuals that are no byte (a few;
    more than the exception list holds, which kernel T defers), values beyond 2^21 (deferred by the wavefront) and one
    extreme spike.  `malformed` is a plain tile whose payload is cut short (see _payloads)."""
    rng = np.random.default_rng(100 + k)
    v = oracle.terrain_i32(3000 + 211 * k, 500 + 97 * k, tr, tc).copy()
    if kind == "few":
        v += ((rng.random((tr, tc)) < 0.0005) * rng.integers(-5000, 5000, (tr, tc))).astype(np.int32)
    elif kind == "many":
        v += ((rng.random((tr, tc)) < 0.02) * rng.integers(-5000, 5000, (tr, tc))).astype(np.int32)
    elif kind == "range":
        v *= 500
    elif kind == "spike":
        v[90, 100] = -(2 ** 31) + 5
    return v


def _batch(g4, payloads, band):
    """A TileBatch over given payloads, 8-byte aligned back to back."""
    offs, pos = [], 0
    for p in payloads:
        offs.append(pos)
        pos += (len(p) + 7) & ~7
    arena = np.zeros(pos + 8, np.uint8)
    for o, p in zip(offs, payloads):
        arena[o:o + len(p)] = np.frombuffer(p, np.uint8)
    lens = np.array([len(p) for p in payloads], np.uint32)
    return g4.TileBatch(arena, np.array(offs, np.uint64), lens, None, None, None, pos, band)


def _to_device(g4, batch):
    import torch

    return g4.TileBatch(torch.from_numpy(batch.arena).cuda(), torch.from_numpy(batch.offsets.astype(np.int64)).cuda(),
                        torch.from_numpy(batch.lens.astype(np.int32)).cuda(), None, None, None, batch.total_bytes, batch.band)


def _decode(g4, master, batch, device, out=None):
    """Decodes the batch; returns (raster as numpy, status as numpy).  A malformed tile raises FormatError after the
    whole band was decoded."""
    import torch

    b = _to_device(g4, batch) if device else batch
    o = torch.from_numpy(out).cuda() if (device and out is not None) else out
    try:
        r = master.decodeTiles(b, out=o)
    except g4.FormatError:
        r = o if o is not None else None
    st = master.lastStatus.cpu().numpy() if device else np.asarray(master.lastStatus)
    if r is None:
        return None, st
    return (r.cpu().numpy() if device else r), st


@pytest.fixture(scope="module")
def kind_payloads(g4, oracle):
    """kind -> (tile, payload): the oracle's LSOP12 packing of each kind (the malformed one cut to half its length)."""
    out = {}
    for k, kind in enumerate(KINDS):
        tile = _kind_tile(oracle, kind, k)
        p = oracle.master_encode_i32([oracle.CODEC_LSOP12], tile)
        assert p[0] == 0  # codec index 0 = LSOP12
        if kind == "malformed":
            p = p[:len(p) // 2]
        out[kind] = (tile, p)
    return out


@pytest.mark.parametrize("device", [False, True])
def test_every_ordered_pair_of_tile_kinds(g4, oracle, kind_payloads, device):
    """Each ordered pair of kinds as a 1x2 band of 180x240 (W 16, one pair per band)."""
    master = _master(g4)
    band = master._band((180, 480), np.int32, 180, 240)
    for a, b in itertools.product(KINDS, KINDS):
        (ta, pa), (tb, pb) = kind_payloads[a], kind_payloads[b]
        raster, st = _decode(g4, master, _batch(g4, [pa, pb], band), device, out=np.zeros((180, 480), np.int32))
        want_st = [G4_ERR_FORMAT if k == "malformed" else G4_OK for k in (a, b)]
        assert list(st) == want_st, "%s + %s: status %s" % (a, b, list(st))
        for k, (kind, t) in enumerate(((a, ta), (b, tb))):
            if kind != "malformed":
                assert np.array_equal(raster[:, 240 * k:240 * (k + 1)], t), "%s + %s: tile %d (%s)" % (a, b, k, kind)


# (tile rows, tile columns): W 4 pairs (15 and 11 strips), W 8 pairs (15 and 16), W 16 pairs (15 and 16), single-tile
# controls at 512 columns (W 16, 32 strips) and 100 columns (W 4, 25 strips: no W gives 16 strips or fewer)
SHAPES = [(60, 60), (64, 44), (90, 120), (128, 128), (180, 240), (256, 256), (512, 512), (90, 100)]


@pytest.mark.parametrize("shape", SHAPES)
def test_band_shapes_and_odd_tile_counts(g4, oracle, shape):
    """Bands of 1, 2, 3 and 7 tiles: odd counts leave the second half of the last warp without a tile."""
    tr, tc = shape
    master = _master(g4)
    for n in (1, 2, 3, 7):
        grid = oracle.terrain_i32(400 * n, 900 + tc, tr, n * tc)
        batch = master.encodeTiles(grid, tr, tc)
        for t in range(n):
            assert batch.payload(t) == oracle.master_encode_i32([oracle.CODEC_LSOP12], grid[:, t * tc:(t + 1) * tc]), \
                "%s n=%d tile %d" % (shape, n, t)
        assert np.array_equal(master.decodeTiles(batch), grid), "%s n=%d" % (shape, n)


def test_tile_list_with_permuted_tiles(g4, oracle, kind_payloads):
    """A tile-list decode whose list positions map to scattered, non-adjacent places in memory in permuted order, so
    the tiles of a warp are neither neighbours in the output nor in the list's natural order."""
    import torch

    kinds = ["plain", "few", "range", "plain", "many", "spike", "plain", "few", "plain"]
    perm = [5, 2, 8, 0, 7, 3, 1, 6, 4]
    tr, tc, pitch = 180, 240, 256
    master = _master(g4)
    payloads = [kind_payloads[k][1] for k in kinds]
    b = _batch(g4, payloads, None)
    refs = [(perm[k] * 2 * tr * pitch + 64, pitch) for k in range(len(kinds))]  # a gap of one tile between slots
    n = len(kinds) * 2 * tr * pitch + 128
    for device in (False, True):
        out = np.full(n, -7, np.int32)
        if device:
            dev = torch.from_numpy(out).cuda()
            master.decodeTileList(torch.from_numpy(b.arena).cuda(), torch.from_numpy(b.offsets.astype(np.int64)).cuda(),
                                  torch.from_numpy(b.lens.astype(np.int32)).cuda(), dev, refs, tr, tc)
            out = dev.cpu().numpy()
        else:
            master.decodeTileList(b.arena, b.offsets, b.lens, out, refs, tr, tc)
        touched = np.zeros(n, bool)
        for k, (off, p) in enumerate(refs):
            v = out[off:off + tr * p].reshape(tr, p)
            assert np.array_equal(v[:, :tc], kind_payloads[kinds[k]][0]), "device=%s tile %d (%s)" % (device, k, kinds[k])
            for r in range(tr):
                touched[off + r * p:off + r * p + tc] = True
        assert np.all(out[~touched] == -7), "device=%s: cells outside the tiles were written" % device


@pytest.mark.parametrize("extra", [8, 4])
def test_band_inside_a_wider_raster(g4, oracle, kind_payloads, extra):
    """grid_pitch > band width: extra = 8 keeps the 256-bit raster stores, extra = 4 (a pitch that is no multiple of 8
    samples) takes the 128-bit ones.  Three tiles per row: one pair and one lone tile per band row."""
    kinds = ["plain", "many", "few", "spike", "malformed", "range"]
    tr, tc = 180, 240
    master = _master(g4)
    band = master._band((2 * tr, 3 * tc), np.int32, tr, tc)
    band.grid_pitch = 3 * tc + extra
    batch = _batch(g4, [kind_payloads[k][1] for k in kinds], band)
    for device in (False, True):
        out = np.full((2 * tr, 3 * tc + extra), -9, np.int32)
        raster, st = _decode(g4, master, batch, device, out=out)
        assert list(st) == [G4_ERR_FORMAT if k == "malformed" else G4_OK for k in kinds], "device=%s" % device
        for t, kind in enumerate(kinds):
            if kind == "malformed":
                continue
            r0, c0 = (t // 3) * tr, (t % 3) * tc
            assert np.array_equal(raster[r0:r0 + tr, c0:c0 + tc], kind_payloads[kind][0]), "device=%s tile %d (%s)" % (device, t, kind)
        assert np.all(raster[:, 3 * tc:] == -9), "device=%s: the columns past the band were written" % device


def test_mixed_codec_band(g4, oracle):
    """LSOP12 tiles beside tiles that other codecs win (constant and noise tiles), so that the tiles of a pair are
    neighbours in the LSOP list but not in the band."""
    tr, tc = 90, 120
    rng = np.random.default_rng(17)
    master = _master(g4, ("GvrsHuffman", "GvrsDeflate", "LSOP12"))
    ids = [oracle.CODEC_HUFFMAN, oracle.CODEC_DEFLATE, oracle.CODEC_LSOP12]
    grid = oracle.terrain_i32(5000, 7000, 3 * tr, 5 * tc).copy()
    for t in (1, 4, 7, 8, 12):
        r0, c0 = (t // 5) * tr, (t % 5) * tc
        if t % 2:
            grid[r0:r0 + tr, c0:c0 + tc] = 1234 + t
        else:
            grid[r0:r0 + tr, c0:c0 + tc] = rng.integers(-(2 ** 31), 2 ** 31, (tr, tc), dtype=np.int64).astype(np.int32)
    batch = master.encodeTiles(grid, tr, tc)
    codecs = set()
    for t in range(15):
        r0, c0 = (t // 5) * tr, (t % 5) * tc
        p = batch.payload(t)
        assert p == oracle.master_encode_i32(ids, grid[r0:r0 + tr, c0:c0 + tc]), "tile %d" % t
        codecs.add(p[0])
    assert 2 in codecs and len(codecs) >= 2, codecs  # LSOP12 and at least one other codec (or raw)
    assert np.array_equal(master.decodeTiles(batch), grid)
    import torch

    dbatch = master.encodeTiles(torch.from_numpy(grid).cuda(), tr, tc)
    assert np.array_equal(master.decodeTiles(dbatch).cpu().numpy(), grid)
