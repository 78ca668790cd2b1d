"""-m gpu: CodecHuffman CUDA path vs the CPU oracle (byte-exact streams, bit-exact decoded grids)."""
import numpy as np
import pytest

from gpu_common import first_diff, parity_grids

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def g4():
    import gridfour_b200

    return gridfour_b200


def test_encode_streams_byte_exact(g4, oracle):
    codec = g4.CodecHuffman()
    for name, grid in parity_grids(oracle).items():
        exp, pred = oracle.codec_encode_i32(oracle.CODEC_HUFFMAN, 3, grid)
        got = codec.encode(3, grid.shape[0], grid.shape[1], grid)
        assert got is not None, name
        assert codec.lastPredictor == pred, (name, codec.lastPredictor, pred)
        assert got == exp, "%s: %s" % (name, first_diff(got, exp))


def test_decode_bit_exact(g4, oracle):
    codec = g4.CodecHuffman()
    for name, grid in parity_grids(oracle).items():
        packing, _ = oracle.codec_encode_i32(oracle.CODEC_HUFFMAN, 0, grid)
        out = codec.decode(grid.shape[0], grid.shape[1], packing)
        assert np.array_equal(out, grid), "%s: %s" % (name, first_diff(out, grid))


@pytest.mark.parametrize("pred", [1, 2, 3])
def test_decode_every_predictor(g4, oracle, pred):
    """The encoder picks one predictor per tile; force each one through the decoder."""
    codec = g4.CodecHuffman()
    for name in ("terrain90x120", "terrain61x77", "wide", "two_by_two"):
        grid = parity_grids(oracle)[name]
        n, seed, m32 = oracle.predictor_encode(pred, grid)
        text, nbits = oracle.huffman_encode(np.frombuffer(m32, np.uint8))
        hdr = bytes([0, pred]) + int(seed).to_bytes(4, "little", signed=True) + int(n).to_bytes(4, "little")
        packing = hdr + text
        ref = oracle.codec_decode_i32(oracle.CODEC_HUFFMAN, grid.shape[0], grid.shape[1], packing)
        assert np.array_equal(ref, grid)
        out = codec.decode(grid.shape[0], grid.shape[1], packing)
        assert np.array_equal(out, grid), "%s pred %d: %s" % (name, pred, first_diff(out, grid))


def test_malformed_packing_is_an_io_error(g4, oracle):
    codec = g4.CodecHuffman()
    grid = parity_grids(oracle)["terrain45x60"]
    packing, _ = oracle.codec_encode_i32(oracle.CODEC_HUFFMAN, 0, grid)
    bad = bytearray(packing)
    bad[1] = 9  # unknown predictor -> IOException("Unknown PredictorCorrector type")
    with pytest.raises(IOError):
        codec.decode(45, 60, bytes(bad))
    with pytest.raises(IOError):
        codec.decode(45, 60, packing[:40])  # truncated text


def test_batch_encode_decode_host(g4, oracle):
    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("GvrsHuffman", g4.CodecHuffman)
    master = g4.CodecMaster(spec)
    grid = oracle.terrain_i32(5000, 9000, 4 * 90, 3 * 120)
    rng = np.random.default_rng(0)
    grid[90:180, 120:240] = rng.integers(-(2 ** 31), 2 ** 31, (90, 120), dtype=np.int64).astype(np.int32)  # raw tile
    batch = master.encodeTiles(grid, 90, 120)
    assert batch.lens.size == 12
    for t in range(12):
        tr, tc = divmod(t, 3)
        tile = grid[tr * 90:(tr + 1) * 90, tc * 120:(tc + 1) * 120]
        exp = oracle.master_encode_i32([0], tile)
        got = batch.payload(t)
        assert got == exp, "tile %d: %s" % (t, first_diff(got, exp))
        assert int(batch.offsets[t]) % 8 == 0
    assert batch.codec[4] == 255 and batch.lens[4] == 90 * 120 * 4
    out = master.decodeTiles(batch)
    assert np.array_equal(out, grid), first_diff(out, grid)


def test_batch_device_path_matches_host_path(g4, oracle):
    import torch

    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("GvrsHuffman", g4.CodecHuffman)
    master = g4.CodecMaster(spec)
    grid = oracle.terrain_i32(0, 0, 2 * 180, 2 * 240)
    hb = master.encodeTiles(grid, 180, 240)
    dgrid = torch.from_numpy(grid).cuda()
    db = master.encodeTiles(dgrid, 180, 240)
    assert db.total_bytes == hb.total_bytes
    assert np.array_equal(db.lens.cpu().numpy().astype(np.uint32), hb.lens)
    assert np.array_equal(db.arena[: db.total_bytes].cpu().numpy(), hb.arena)
    out = master.decodeTiles(db)
    assert torch.equal(out, dgrid)
    for t in range(4):
        tr, tc = divmod(t, 2)
        tile = grid[tr * 180:(tr + 1) * 180, tc * 240:(tc + 1) * 240]
        assert hb.payload(t) == oracle.master_encode_i32([0], tile)


def test_terrain_generator_matches_cpu(g4, oracle):
    import torch

    ctx = g4.Context.default()
    t = torch.empty((97, 131), dtype=torch.int32, device="cuda")
    ctx.fill_terrain(t.data_ptr(), 0, 12345, 67890, 97, 131)
    ctx.synchronize()
    assert np.array_equal(t.cpu().numpy(), oracle.terrain_i32(12345, 67890, 97, 131))
    f = torch.empty((33, 65), dtype=torch.float32, device="cuda")
    ctx.fill_terrain(f.data_ptr(), 1, 5, 7, 33, 65)
    ctx.synchronize()
    assert np.array_equal(f.cpu().numpy(), oracle.terrain_f32(5, 7, 33, 65))


def test_general_decoder_unaligned_packings(g4, oracle):
    """huffman_decode_kernel stages a packing in shared memory (g4_huff_fast.cuh) only when it starts on a 4-byte
    boundary; any other packing goes through the general decoder over HBM (g4_huffdec.cuh).  Every parity grid's packing
    sits at arena offsets 1, 2 and 3 (mod 4) of one tile-list call and decodes bit-exact at each.  Triangle tiles take
    the fused kernel (g4_huff2.cuh) whatever their alignment; the oversized packings below send them to the general one."""
    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("GvrsHuffman", g4.CodecHuffman)
    master = g4.CodecMaster(spec)
    longer_than_raw = []
    for name, grid in parity_grids(oracle).items():
        R, C = grid.shape
        packing, _ = oracle.codec_encode_i32(oracle.CODEC_HUFFMAN, 0, grid)
        if len(packing) >= 4 * grid.size:  # a tile list reads such a payload as a raw tile or rejects it (CodecMaster never writes one)
            longer_than_raw.append(name)
            continue
        arena = np.zeros(3 * (len(packing) + 32), np.uint8)
        offsets, pos = [], 0
        for mis in (1, 2, 3):
            pos = (pos + 15) // 16 * 16 + mis
            arena[pos:pos + len(packing)] = np.frombuffer(packing, np.uint8)
            offsets.append(pos)
            pos += len(packing)
        out = np.full(3 * grid.size, -7, np.int32)
        refs = [(k * grid.size, C) for k in range(3)]
        master.decodeTileList(arena, np.array(offsets, np.uint64), np.full(3, len(packing), np.uint32), out, refs, R, C)
        assert not master.lastStatus.any(), (name, master.lastStatus)
        for k, mis in enumerate((1, 2, 3)):
            got = out[k * grid.size:(k + 1) * grid.size].reshape(R, C)
            assert np.array_equal(got, grid), "%s at offset %d mod 4: %s" % (name, mis, first_diff(got, grid))
    assert longer_than_raw == ["noise"]  # its kind of content (multi-byte M32 codes) is among the oversized grids below


@pytest.mark.parametrize("pred", [3, 1, 2])
def test_general_decoder_oversized_packings(g4, oracle, pred):
    """A packing larger than both staging buffers -- the fused Triangle kernel's (n*6/8 + 256 bytes, at least 32 rows of
    the tile) and huffman_decode_kernel's (n*6/8 + 64 bytes, at least 8 KB) -- goes through the general decoder over HBM,
    whatever the predictor.  One grid per predictor: the noise is the predictor's residual, 1 % of it full-range (the
    multi-byte M32 codes of a random raster)."""
    R, C = 180, 240
    rng = np.random.default_rng(5 + pred)
    noise = rng.integers(-300, 301, (R, C), dtype=np.int64)
    tail = rng.random((R, C)) < 0.01
    noise[tail] = rng.integers(-(2 ** 31), 2 ** 31, int(tail.sum()), dtype=np.int64)
    if pred == 3:  # Triangle: a 2-D cumulative sum
        grid = noise.cumsum(axis=0).cumsum(axis=1)
    elif pred == 1:  # Differencing: a row cumulative sum
        grid = noise.cumsum(axis=1)
    else:  # Linear: a second row cumulative sum
        grid = noise.cumsum(axis=1).cumsum(axis=1)
    grid = grid.astype(np.int32)  # wraps like the codec's 32-bit arithmetic
    packing, best = oracle.codec_encode_i32(oracle.CODEC_HUFFMAN, 0, grid)
    assert best == pred
    n = grid.size
    assert len(packing) > max(n * 6 // 8 + 256, 32 * C * 4, 8192 + 8), len(packing)
    out = g4.CodecHuffman().decode(R, C, packing)
    assert np.array_equal(out, grid), first_diff(out, grid)
