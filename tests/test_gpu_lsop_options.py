"""The LSOP12 encoder's two switches (lsop/LsEncoder12.java:93-119): the Deflate alternative (on by default) and the value
checksum (off by default).  Every packing is compared byte for byte with the oracle's LsEncoder12 restatement
(oracle.lsop12_encode(..., deflate=, checksum=)); batches are compared with the CodecMaster rule applied here to the oracle's
per-codec packings; checksummed packings are decoded and checked on the GPU; the option bits of the C ABI are checked for
what they accept and reject."""
import ctypes as C
import warnings

import numpy as np
import pytest

G4_OK, G4_ERR_ARG, G4_CHECKSUM_MISMATCH = 0, -1, 2
G4_CODEC_HUFFMAN, G4_CODEC_DEFLATE, G4_CODEC_LSOP12 = 0, 1, 4
G4_LSOP12_NO_DEFLATE, G4_LSOP12_VALUE_CHECKSUM = 1 << 8, 1 << 9
G4_CODEC_RAW = 255
INT_MIN = -(2 ** 31)
COMBOS = [(True, False), (True, True), (False, False), (False, True)]  # (deflate, checksum)


@pytest.fixture(scope="module")
def g4():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gridfour_b200

    return gridfour_b200


def _enc(g4, deflate, checksum):
    e = g4.LsEncoder12()
    e.setDeflateEnabled(deflate)
    e.setValueChecksumEnabled(checksum)
    return e


def _repetitive(rows, cols, seed):
    """A short random pattern repeated: the M32 streams repeat too, so the level-6 zlib streams beat canonical Huffman."""
    rng = np.random.default_rng(seed)
    return np.tile(rng.integers(-3000, 3000, (6, 10)), (rows // 6 + 1, cols // 10 + 1))[:rows, :cols].astype(np.int32)


def _tiles(oracle):
    rng = np.random.default_rng(11)
    t = {}
    t["terrain90x120"] = oracle.terrain_i32(0, 0, 90, 120)
    t["terrain120x120"] = oracle.terrain_i32(500, 800, 120, 120)
    t["terrain180x240"] = oracle.terrain_i32(7000, 3000, 180, 240)
    t["noise6x6"] = rng.integers(-500, 500, (6, 6)).astype(np.int32)
    t["terrain61x77"] = oracle.terrain_i32(123, 457, 61, 77)
    t["terrain45x63"] = oracle.terrain_i32(9, 31, 45, 63)
    t["terrain512x512"] = oracle.terrain_i32(2000, 4000, 512, 512)
    t["repeat90x120"] = _repetitive(90, 120, 1)
    t["repeat64x70"] = _repetitive(64, 70, 2)
    nulls = oracle.terrain_i32(300, 300, 90, 120)
    nulls[10:30, 40:70] = INT_MIN
    nulls[:, 0] = INT_MIN
    t["nulls90x120"] = nulls
    t["fullrange40x40"] = rng.integers(-(2 ** 31), 2 ** 31, (40, 40), dtype=np.int64).astype(np.int32)
    return t


@pytest.mark.gpu
def test_per_tile_packings_equal_the_oracle(g4, oracle):
    tiles = _tiles(oracle)
    deflate_won = []
    for name, tile in tiles.items():
        nr, nc = tile.shape
        for deflate, checksum in COMBOS:
            want = oracle.lsop12_encode(3, tile, deflate=deflate, checksum=checksum)
            got = _enc(g4, deflate, checksum).encode(3, nr, nc, tile)
            assert got == want, (name, deflate, checksum)
            assert (got[1] & 0x80 != 0) == checksum
            if want[1] & 0x0F == 1:
                assert deflate
                deflate_won.append((name, checksum))
    # the relocated checksum (byte 63, behind the two M32 lengths) is exercised
    assert any(c for _n, c in deflate_won) and any(n.startswith("repeat") for n, _c in deflate_won)


@pytest.mark.gpu
def test_too_small_and_singular_tiles_decline_in_every_combination(g4, oracle):
    for tile in (np.arange(5 * 40, dtype=np.int32).reshape(5, 40), np.arange(40 * 5, dtype=np.int32).reshape(40, 5),
                 np.full((20, 20), 17, np.int32)):
        for deflate, checksum in COMBOS:
            assert oracle.lsop12_encode(0, tile, deflate=deflate, checksum=checksum) is None
            assert _enc(g4, deflate, checksum).encode(0, tile.shape[0], tile.shape[1], tile) is None


def _master(g4, deflate, checksum):
    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("GvrsHuffman", g4.CodecHuffman)
    spec.addCompressionCodec("GvrsDeflate", g4.CodecDeflate)
    spec.addCompressionCodec("LSOP12", g4.LsEncoder12, g4.LsDecoder12)
    master = g4.CodecMaster(spec)
    lsop = master.getEncoder("LSOP12")
    lsop.setDeflateEnabled(deflate)
    lsop.setValueChecksumEnabled(checksum)
    return master


def _expected_payload(oracle, tile, deflate, checksum, raw):
    """CodecMaster.encodeSingleThread (strictly smaller wins, ties to the lowest index), then TileElement's raw fallback."""
    packs = [oracle.codec_encode_i32(oracle.CODEC_HUFFMAN, 0, tile)[0], oracle.codec_encode_i32(oracle.CODEC_DEFLATE, 1, tile)[0],
             oracle.lsop12_encode(2, tile, deflate=deflate, checksum=checksum)]
    best = None
    for p in packs:
        if p is not None and (best is None or len(p) < len(best)):
            best = p
    return raw if best is None or len(best) >= len(raw) else best


def _grid(oracle):
    """2 x 4 tiles of 90 x 120: terrain, one repetitive tile (the Deflate form wins), one tile with nulls."""
    g = oracle.terrain_i32(1200, 2400, 180, 480)
    g[0:90, 120:240] = _repetitive(90, 120, 3) + 20000
    g[100:130, 260:330] = INT_MIN
    return g


def _tile_of(g, t, tr, tc, across):
    r, c = divmod(t, across)
    return np.ascontiguousarray(g[r * tr:(r + 1) * tr, c * tc:(c + 1) * tc])


def _check_batch(oracle, batch, codes, tr, tc, deflate, checksum, raw_of):
    across = codes.shape[1] // tc
    n = (codes.shape[0] // tr) * across
    codec = np.asarray(batch.codec.cpu() if hasattr(batch.codec, "cpu") else batch.codec)
    lens = np.asarray(batch.lens.cpu() if hasattr(batch.lens, "cpu") else batch.lens)
    offs = np.asarray(batch.offsets.cpu() if hasattr(batch.offsets, "cpu") else batch.offsets)
    arena = np.asarray(batch.arena.cpu() if hasattr(batch.arena, "cpu") else batch.arena)
    picked_lsop = 0
    for t in range(n):
        tile = _tile_of(codes, t, tr, tc, across)
        want = _expected_payload(oracle, tile, deflate, checksum, raw_of(t, tile))
        got = arena[int(offs[t]):int(offs[t]) + int(lens[t])].tobytes()
        assert got == want, (t, deflate, checksum)
        picked_lsop += int(codec[t] == 2)
        if codec[t] == 2:
            assert (got[1] & 0x80 != 0) == checksum
    return picked_lsop


@pytest.mark.gpu
@pytest.mark.parametrize("deflate,checksum", COMBOS)
def test_batched_encode_follows_the_codec_master_rule(g4, oracle, deflate, checksum):
    import torch

    tr, tc = 90, 120
    g = _grid(oracle)
    master = _master(g4, deflate, checksum)
    raw32 = lambda t, tile: tile.astype("<i4").tobytes()  # noqa: E731
    # host and device memory
    assert _check_batch(oracle, master.encodeTiles(g, tr, tc), g, tr, tc, deflate, checksum, raw32) > 0
    dev = master.encodeTiles(torch.from_numpy(g).cuda(), tr, tc)
    torch.cuda.synchronize()
    assert _check_batch(oracle, dev, g, tr, tc, deflate, checksum, raw32) > 0
    # a short element with a fill value: the codecs see the widened ints, the fill value coded as INT4_NULL_CODE
    s = np.clip(g // 4, -32000, 32000).astype(np.int16)
    s[20:50, 30:90] = -9999
    wide = s.astype(np.int32)
    wide[s == -9999] = INT_MIN

    def raw16(t, tile):
        b = _tile_of(s, t, tr, tc, 4).astype("<i2").tobytes()
        return b + bytes((-len(b)) & 3)

    _check_batch(oracle, master.encodeTiles(s, tr, tc, fillValue=-9999), wide, tr, tc, deflate, checksum, raw16)
    # an integer-coded float band: the codecs see the codes
    icf = g4.IntCodedFloat(10.0, 0.0)
    f = (oracle.terrain_f32(100, 200, 180, 480) / np.float32(7)).astype(np.float32)
    f[5:40, 300:350] = np.nan
    codes = icf.to_int(f)
    _check_batch(oracle, master.encodeTiles(f, tr, tc, icf=icf), codes, tr, tc, deflate, checksum, raw32)
    # a tile list: tiles scattered in a wider raster, each with its own window
    refs = [(r * tr * 480 + c * tc, 480) for r, c in ((1, 3), (0, 1), (1, 0))]
    tl = master.encodeTileList(g, refs, tr, tc)
    for k, (off, _p) in enumerate(refs):
        r, c = divmod(off, 480)
        tile = np.ascontiguousarray(g[r:r + tr, c:c + tc])
        assert tl.payload(k) == _expected_payload(oracle, tile, deflate, checksum, tile.astype("<i4").tobytes()), k


def _lsop_only(g4, deflate, checksum):
    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("LSOP12", g4.LsEncoder12, g4.LsDecoder12)
    master = g4.CodecMaster(spec)
    master.getEncoder("LSOP12").setDeflateEnabled(deflate)
    master.getEncoder("LSOP12").setValueChecksumEnabled(checksum)
    return master


def _cks_pos(p):  # revised header (LsHeader.java:220-245): the two M32 lengths precede the checksum unless the body is canonical
    return 55 if (p[1] & 0x0F) == 2 else 63


@pytest.mark.gpu
@pytest.mark.parametrize("deflate", [True, False])
def test_checksummed_packings_round_trip_and_a_flipped_crc_flags_one_tile(g4, oracle, deflate):
    tr, tc = 90, 120
    g = _grid(oracle)
    master = _lsop_only(g4, deflate, True)
    batch = master.encodeTiles(g, tr, tc)
    assert all(batch.payload(t)[1] & 0x80 for t in range(8) if batch.codec[t] == 0)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        assert np.array_equal(master.decodeTiles(batch), g)
    assert not np.asarray(master.lastStatus).any()
    # short tiles with nulls: decode checks the same widened ints the encoder summed
    s = np.clip(g // 4, -32000, 32000).astype(np.int16)
    s[20:50, 30:90] = -9999
    sb = master.encodeTiles(s, tr, tc, fillValue=-9999)
    want_s = s.copy()
    want_s[s == -9999] = -32768
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        assert np.array_equal(master.decodeTiles(sb), want_s)
    assert not np.asarray(master.lastStatus).any()
    # one flipped CRC byte: that tile alone is flagged, its values are still delivered
    victim = next(t for t in range(8) if batch.codec[t] == 0 and (deflate or batch.payload(t)[1] & 0x0F == 2))
    p = batch.payload(victim)
    arena = np.array(batch.arena, copy=True)
    arena[int(batch.offsets[victim]) + _cks_pos(p)] ^= 0x10
    bad = g4.TileBatch(arena, batch.offsets, batch.lens, batch.codec, batch.predictor, batch.status, batch.total_bytes, batch.band)
    with pytest.warns(g4.ValueChecksumWarning):
        out = master.decodeTiles(bad)
    assert np.array_equal(out, g)
    st = np.asarray(master.lastStatus)
    assert st[victim] == G4_CHECKSUM_MISMATCH and np.count_nonzero(st) == 1


@pytest.mark.gpu
def test_deflate_form_carries_the_checksum_behind_the_lengths(g4, oracle):
    tile = _repetitive(90, 120, 4)
    p = _enc(g4, True, True).encode(0, 90, 120, tile)
    assert p[1] == 0x80 | 0x40 | 1
    assert int.from_bytes(p[63:67], "little") == oracle.crc32c(tile.astype("<i4").tobytes())
    assert np.array_equal(oracle.codec_decode_i32(oracle.CODEC_LSOP12, 90, 120, p), tile)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        assert np.array_equal(g4.LsDecoder12().decode(90, 120, p), tile)


@pytest.mark.gpu
def test_writer_round_trip_with_a_configured_master(g4, oracle):
    from gridfour_b200 import gvrs

    rows, cols = 300, 430
    g = oracle.terrain_i32(50, 60, rows, cols)
    g[0:90, 120:240] = _repetitive(90, 120, 5)
    g[150:170, :] = INT_MIN
    spec = gvrs.GvrsSpec(rows, cols, 90, 120, [gvrs.ElementSpec.integer("z")], ["GvrsHuffman", "GvrsDeflate", "LSOP12"], checksum=True)
    master = _master(g4, True, True)
    w = gvrs.GvrsWriter(spec, uuid=bytes(range(16)), time_modified=1700000000000)
    for name, rid, typ, content, desc in gvrs.codec_metadata(spec.codecs):
        w.add_metadata(name, rid, typ, content, desc)
    w.add_raster(master, g)
    img = gvrs.GvrsImage.parse(w.finish(master._context()))
    reader = g4.CodecMaster(master.spec)  # a master with default encoder options reads the same file
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        assert np.array_equal(img.read_raster(reader, crop=True), g)
    off, lens, _st = img.locate_payloads(reader._context(), 0)
    full = np.full((4 * 90, 4 * 120), INT_MIN, np.int32)
    full[:rows, :cols] = g
    ids = [oracle.CODEC_HUFFMAN, oracle.CODEC_DEFLATE, oracle.CODEC_LSOP12]
    n_cks = 0
    for t in range(16):
        p = img.image[int(off[t]):int(off[t]) + int(lens[t])]
        assert np.array_equal(oracle.master_decode_i32(ids, 90, 120, p), _tile_of(full, t, 90, 120, 4)), t
        n_cks += int(len(p) != 4 * 90 * 120 and p[0] == 2 and p[1] & 0x80 != 0)
    assert n_cks > 0


@pytest.mark.gpu
def test_launch_counts(g4, oracle):
    """Deflate off drops exactly the alternative's launches: M32 sizes, stream offsets, M32 write, the four staged level-6
    zlib kernels of one chunk (sort, match, decide, emit) and the pick.  The checksum adds one launch (the CRC pass)."""
    g = oracle.terrain_i32(0, 0, 180, 240)
    counts = {}
    for deflate, checksum in COMBOS:
        master = _lsop_only(g4, deflate, checksum)
        ctx = master._context()
        master.encodeTiles(g, 90, 120)  # warm: buffers allocated
        n0 = ctx.launch_count
        master.encodeTiles(g, 90, 120)
        counts[(deflate, checksum)] = ctx.launch_count - n0
    assert counts[(True, False)] - counts[(False, False)] == 8
    assert counts[(True, True)] - counts[(True, False)] == 1
    assert counts[(False, True)] - counts[(False, False)] == 1


@pytest.mark.gpu
def test_option_bits_at_the_c_abi(g4, oracle):
    from gridfour_b200 import _lib

    L = _lib.lib()
    ctx = g4.Context.default()
    tile = oracle.terrain_i32(0, 0, 90, 120)
    out = np.empty(90 * 120 * 6 + 1024, np.uint8)
    n = C.c_size_t(0)

    def enc(cid):
        return L.g4_encode_i32(ctx._h, cid, 0, 90, 120, tile.ctypes.data, out.ctypes.data, out.size, C.byref(n), None)

    assert enc(G4_CODEC_LSOP12 | G4_LSOP12_NO_DEFLATE | G4_LSOP12_VALUE_CHECKSUM) == G4_OK
    assert out[:n.value].tobytes() == oracle.lsop12_encode(0, tile, deflate=False, checksum=True)
    assert enc(G4_CODEC_LSOP12 | (1 << 10)) == G4_ERR_ARG
    assert enc(G4_CODEC_LSOP12 | (1 << 30)) == G4_ERR_ARG
    assert enc(G4_CODEC_HUFFMAN | G4_LSOP12_NO_DEFLATE) == G4_ERR_ARG
    assert enc(G4_CODEC_DEFLATE | G4_LSOP12_VALUE_CHECKSUM) == G4_ERR_ARG
    # the name and supported calls take plain ids only
    assert L.g4_codec_name(G4_CODEC_LSOP12 | G4_LSOP12_NO_DEFLATE) is None
    assert L.g4_codec_supported(G4_CODEC_LSOP12 | G4_LSOP12_VALUE_CHECKSUM, 1) == 0
    assert L.g4_codec_supported(G4_CODEC_LSOP12 | G4_LSOP12_VALUE_CHECKSUM, 0) == 0
    # per-tile decode ignores the bits
    pk = np.frombuffer(oracle.lsop12_encode(0, tile, checksum=True), np.uint8)
    dec = np.empty((90, 120), np.int32)
    assert L.g4_decode_i32(ctx._h, G4_CODEC_LSOP12 | G4_LSOP12_VALUE_CHECKSUM, 90, 120, pk.ctypes.data, pk.size, dec.ctypes.data) == G4_OK
    assert np.array_equal(dec, tile)
    assert L.g4_decode_i32(ctx._h, G4_CODEC_LSOP12 | (1 << 11), 90, 120, pk.ctypes.data, pk.size, dec.ctypes.data) == G4_ERR_ARG
    # batched: a list with bad bits is refused by encode and decode; a list with the bits decodes and analyzes as without
    g = _grid(oracle)
    master = _master(g4, False, True)
    batch = master.encodeTiles(g, 90, 120)
    cl_bits = master._native_list()
    assert cl_bits.codec_ids[2] == G4_CODEC_LSOP12 | G4_LSOP12_NO_DEFLATE | G4_LSOP12_VALUE_CHECKSUM
    cl_plain = master.spec.native_list()
    grid = np.empty_like(g)
    status = np.empty(8, np.int32)
    arena = np.ascontiguousarray(batch.arena)
    off = np.ascontiguousarray(batch.offsets, np.uint64)
    ln = np.ascontiguousarray(batch.lens, np.uint32)

    def decode(cl):
        grid[...] = 0
        return L.g4_decode_tiles_bounded(ctx._h, C.byref(cl), C.byref(batch.band), 0, arena.ctypes.data, arena.size, off.ctypes.data,
                                         ln.ctypes.data, grid.ctypes.data, status.ctypes.data)

    assert decode(cl_bits) == G4_OK and np.array_equal(grid, g)
    assert decode(cl_plain) == G4_OK and np.array_equal(grid, g)
    for bad_entry in (G4_CODEC_LSOP12 | (1 << 12), G4_CODEC_DEFLATE | G4_LSOP12_NO_DEFLATE):
        cl_bad = master._native_list()
        cl_bad.codec_ids[2 if bad_entry & 0xFF == G4_CODEC_LSOP12 else 1] = bad_entry
        assert decode(cl_bad) == G4_ERR_ARG
        tot = C.c_uint64(0)
        cap = int(L.g4_encode_arena_bound(C.byref(batch.band)))
        a2 = np.empty(cap, np.uint8)
        o2, l2, c2, p2, s2 = np.empty(8, np.uint64), np.empty(8, np.uint32), np.empty(8, np.uint8), np.empty(8, np.uint8), np.empty(8, np.int32)
        assert L.g4_encode_tiles(ctx._h, C.byref(cl_bad), C.byref(batch.band), 0, g.ctypes.data, a2.ctypes.data, cap, o2.ctypes.data,
                                 l2.ctypes.data, c2.ctypes.data, p2.ctypes.data, s2.ctypes.data, C.byref(tot)) == G4_ERR_ARG
    s_bits = g4.analyze_tiles(ctx, cl_bits, batch.band, arena, off, ln)
    s_plain = g4.analyze_tiles(ctx, cl_plain, batch.band, arena, off, ln)
    assert [bytes(x) for x in s_bits] == [bytes(x) for x in s_plain]
