"""Integer-coded float elements on the GPU: g4_icf_map, g4_encode_tiles_icf and g4_decode_tiles_icf against the CPU oracle
(oracle/g4o_icf.cpp for the mapping, the oracle's codecs for the payloads), the reference's four ICF sample files, the GVRS
writer and reader, and the tile cache's float accessors."""
import ctypes as C

import numpy as np
import pytest

from gvrs_common import sample_files

G4_OK, G4_ERR_ARG, G4_ERR_FORMAT = 0, -1, -2
G4_ELEM_I32, G4_ELEM_ICF = 0, 3
G4_MEM_HOST, G4_MEM_DEVICE = 0, 1
INT_MIN = -(2 ** 31)
ORACLE_IDS = {"GvrsHuffman": 0, "GvrsDeflate": 1, "GvrsFloat": 2, "LSOP12": 4}


@pytest.fixture(scope="module")
def g4():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gridfour_b200

    return gridfour_b200


@pytest.fixture(scope="module")
def icf_ref():
    from oracle import g4icf

    return g4icf


def _master(g4, codecs):
    if codecs is None:
        return g4.CodecMaster()
    spec = g4.CodecSpecification(default=False)
    classes = {"GvrsHuffman": (g4.CodecHuffman,), "GvrsDeflate": (g4.CodecDeflate,), "GvrsFloat": (g4.CodecFloat,),
               "LSOP12": (g4.LsEncoder12, g4.LsDecoder12)}
    for c in codecs:
        spec.addCompressionCodec(c, *classes[c])
    return g4.CodecMaster(spec)


def _ids(master):
    return [ORACLE_IDS[c[0]] for c in master.spec.codecList]


def _bits_input(rng, rows, cols):
    """Random float32 bit patterns with the adversarial values spliced in (NaN payloads, infinities, ties, saturation)."""
    v = rng.integers(0, 2 ** 32, rows * cols, dtype=np.uint64).astype(np.uint32).view(np.float32)
    special = np.array([np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0, 0.5, -0.5, 2.5, -2.5, np.float32(0.49999997), 3e9, -3e9,
                        1e-45, -1e-45, 3.4028235e38, -3.4028235e38, 16777217.0, -11000.5, 123.45], np.float32)
    special = np.concatenate([special, np.array([0x7FC12345, 0xFF800001], np.uint32).view(np.float32)])
    with np.errstate(invalid="ignore"):
        special = np.concatenate([special, special / np.float32(3)])[:v.size]
    v[:special.size] = special
    return v.reshape(rows, cols)


@pytest.mark.gpu
@pytest.mark.parametrize("device", [False, True])
def test_icf_map_equals_oracle(g4, icf_ref, device):
    import torch

    rng = np.random.default_rng(11)
    for scale, offset, fill_int, fill_value in [(1.0, 0.0, INT_MIN, np.nan), (1000.0, -0.5, INT_MIN, np.nan),
                                                (np.float32(0.1), -11000.5, -7, -1.5), (-2.0, 3.0, 0, np.inf)]:
        icf = g4.IntCodedFloat(scale, offset, fill_int, fill_value)
        for rows, cols in [(1, 1), (3, 5), (17, 33), (64, 256), (9, 1021)]:
            values = _bits_input(rng, rows, cols)
            codes = rng.integers(INT_MIN, 2 ** 31, (rows, cols), dtype=np.int64).astype(np.int32)
            codes.flat[::7] = fill_int
            want_k = icf_ref.icf_to_int(values, scale, offset, fill_int)
            want_f = icf_ref.icf_to_float(codes, scale, offset, fill_int, fill_value)
            for off in range(4):
                pitch = cols + (off * 3 + 1) % 4   # row pitches at every residue mod 4 across the offsets
                big_v = np.zeros((rows, pitch + 4), np.float32)
                big_k = np.zeros((rows, pitch + 4), np.int32)
                big_v[:, off:off + cols] = values
                big_k[:, off:off + cols] = codes
                if device:
                    src_v = torch.from_numpy(big_v).cuda()[:, off:off + cols]
                    src_k = torch.from_numpy(big_k).cuda()[:, off:off + cols]
                else:
                    src_v, src_k = big_v[:, off:off + cols], big_k[:, off:off + cols]
                got_k = icf.to_int(src_v)
                got_f = icf.to_float(src_k)
                if device:
                    torch.cuda.synchronize()
                    got_k, got_f = got_k.cpu().numpy(), got_f.cpu().numpy()
                assert np.array_equal(got_k.view(np.uint32), want_k.view(np.uint32)), (scale, rows, cols, off)
                assert np.array_equal(got_f.view(np.uint32), want_f.view(np.uint32)), (scale, rows, cols, off)
                # in place: the destination is the source buffer
                if device:
                    t = torch.from_numpy(big_k).cuda()
                    icf.to_float(t[:, off:off + cols], out=t[:, off:off + cols].view(torch.float32))
                    torch.cuda.synchronize()
                    inplace = t.cpu().numpy()
                else:
                    inplace = big_k.copy()
                    icf.to_float(inplace[:, off:off + cols], out=inplace[:, off:off + cols].view(np.float32))
                assert np.array_equal(inplace[:, off:off + cols].view(np.uint32), want_f.view(np.uint32))
                assert np.array_equal(inplace[:, :off], big_k[:, :off]) and np.array_equal(inplace[:, off + cols:], big_k[:, off + cols:])


@pytest.mark.gpu
def test_icf_map_arguments(g4):
    from gridfour_b200 import _lib

    L = _lib.lib()
    ctx = g4.Context.default()
    a = np.zeros((2, 4), np.float32)
    b = np.zeros((2, 4), np.int32)
    for scale in [0.0, float("inf"), float("nan")]:
        d = _lib.IcfDesc(scale, 0.0, INT_MIN, float("nan"))
        assert L.g4_icf_map(ctx._h, 0, C.byref(d), G4_MEM_HOST, 2, 4, a.ctypes.data, 4, b.ctypes.data, 4) == G4_ERR_ARG
    assert L.g4_icf_map(ctx._h, 0, None, G4_MEM_HOST, 2, 4, a.ctypes.data, 4, b.ctypes.data, 4) == G4_ERR_ARG
    d = _lib.IcfDesc(1.0, 0.0, INT_MIN, float("nan"))
    assert L.g4_icf_map(ctx._h, 0, C.byref(d), G4_MEM_HOST, 2, 4, a.ctypes.data, 3, b.ctypes.data, 4) == G4_ERR_ARG
    assert L.g4_icf_map(ctx._h, 0, C.byref(d), G4_MEM_HOST, 2, 4, a.ctypes.data, 4, b.ctypes.data, 4) == G4_OK


def _raster(oracle, scale):
    """3 x 4 tiles of 90 x 120: decimetre terrain with NaN holes and one tile of wide-range noise whose codes fall back to raw."""
    f = oracle.terrain_f32(300, 700, 270, 480)
    f[10:40, 50:200] = np.nan
    f[200:205, :] = np.nan
    rng = np.random.default_rng(5)
    f[90:180, 240:360] = rng.uniform(-2e8, 2e8, (90, 120)).astype(np.float32) / np.float32(scale)
    return f


@pytest.mark.gpu
@pytest.mark.parametrize("codecs", [["GvrsHuffman", "GvrsDeflate"], ["LSOP12"], None], ids=["huff_deflate", "lsop12", "default"])
@pytest.mark.parametrize("device", [False, True])
def test_encode_tiles_icf_equals_int_encode_of_mapped_codes(g4, oracle, icf_ref, codecs, device):
    import torch

    icf = g4.IntCodedFloat(10.0, 0.0)
    f = _raster(oracle, 10.0)
    codes = icf_ref.icf_to_int(f, 10.0, 0.0)
    master = _master(g4, codecs)
    if device:
        got = master.encodeTiles(torch.from_numpy(f).cuda(), 90, 120, icf=icf)
        want = master.encodeTiles(torch.from_numpy(codes).cuda(), 90, 120)
        torch.cuda.synchronize()
        host = lambda x: x.cpu().numpy()  # noqa: E731
    else:
        got = master.encodeTiles(f, 90, 120, icf=icf)
        want = master.encodeTiles(codes, 90, 120)
        host = np.asarray
    assert got.icf == icf and got.total_bytes == want.total_bytes
    for name in ["offsets", "lens", "codec", "predictor", "status"]:
        assert np.array_equal(host(getattr(got, name)), host(getattr(want, name))), name
    assert np.array_equal(host(got.arena)[:got.total_bytes], host(want.arena)[:want.total_bytes])
    lens, codec = host(got.lens), host(got.codec)
    assert codec[1 * 4 + 2] == 255 and lens[1 * 4 + 2] == 4 * 90 * 120  # the noise tile is stored raw: its codes
    arena, off = host(got.arena), host(got.offsets)
    ref_arena, slot, ref_lens = oracle.encode_grid(_ids(master), codes, 90, 120)
    for t in [0, 1, 5, 6, 11]:
        assert np.array_equal(lens[t], ref_lens[t]), t
        assert bytes(arena[int(off[t]):int(off[t]) + int(lens[t])]) == bytes(ref_arena[t * slot:t * slot + int(ref_lens[t])]), t


def _decode_icf(g4, master, batch, icf, mem, arena, arena_len, offsets, lens, grid, status, band=None):
    from gridfour_b200 import _lib

    d = icf.desc()
    cl = master.spec.native_list()
    return _lib.lib().g4_decode_tiles_icf(master._context()._h, C.byref(cl), C.byref(band or batch.band), C.byref(d), mem, arena,
                                          arena_len, offsets, lens, grid, status)


@pytest.mark.gpu
@pytest.mark.parametrize("device", [False, True])
def test_decode_tiles_icf(g4, oracle, icf_ref, device):
    import torch

    from gridfour_b200 import _lib

    icf = g4.IntCodedFloat(10.0, 0.0)
    f = _raster(oracle, 10.0)
    master = _master(g4, ["GvrsHuffman", "GvrsDeflate", "LSOP12"])
    ctx = master._context()
    batch = master.encodeTiles(torch.from_numpy(f).cuda() if device else f, 90, 120, icf=icf)
    as_int = g4.TileBatch(batch.arena, batch.offsets, batch.lens, None, None, None, batch.total_bytes, batch.band)
    as_int.band = _lib.BandDesc(*[getattr(batch.band, n) for n, _ in _lib.BandDesc._fields_])
    as_int.band.elem_type = G4_ELEM_I32
    n0 = ctx.launch_count
    codes = master.decodeTiles(as_int)
    n1 = ctx.launch_count
    got = master.decodeTiles(batch)
    n2 = ctx.launch_count
    if device:
        torch.cuda.synchronize()
        codes, got = codes.cpu().numpy(), got.cpu().numpy()
        assert n2 - n1 == n1 - n0 + 1
    assert got.dtype == np.float32
    want = icf_ref.icf_to_float(codes, 10.0, 0.0)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(codes, icf_ref.icf_to_int(f, 10.0, 0.0))

    # a band inside a wider raster: the columns outside it are never written
    band = _lib.BandDesc(*[getattr(batch.band, n) for n, _ in _lib.BandDesc._fields_])
    band.grid_pitch = 480 + 13
    wide = np.full((270, 493), 7.25, np.float32)
    status = np.zeros(12, np.int32)
    if device:
        wd, sd = torch.from_numpy(wide).cuda(), torch.from_numpy(status).cuda()
        ctx.after_torch_stream(wd.device)
        st = _decode_icf(g4, master, batch, icf, G4_MEM_DEVICE, batch.arena.data_ptr(), int(batch.arena.numel()), batch.offsets.data_ptr(),
                         batch.lens.data_ptr(), wd.data_ptr(), sd.data_ptr(), band)
        ctx.synchronize()
        out, status = wd.cpu().numpy(), sd.cpu().numpy()
    else:
        out = wide.copy()
        a = np.ascontiguousarray(batch.arena)
        st = _decode_icf(g4, master, batch, icf, G4_MEM_HOST, a.ctypes.data, a.size, batch.offsets.ctypes.data, batch.lens.ctypes.data,
                         out.ctypes.data, status.ctypes.data, band)
    assert st == G4_OK and not status.any()
    assert np.array_equal(out[:, :480].view(np.uint32), want.view(np.uint32))
    assert (out[:, 480:] == 7.25).all()

    # an out-of-arena directory entry: G4_ERR_FORMAT on that tile only
    off = (batch.offsets.cpu().numpy() if device else np.array(batch.offsets)).astype(np.uint64)
    ln = (batch.lens.cpu().numpy() if device else np.array(batch.lens)).astype(np.uint32)
    off[7] = batch.total_bytes + 64
    out = np.zeros((270, 480), np.float32)
    status = np.zeros(12, np.int32)
    if device:
        od, ld, gd, sd = (torch.from_numpy(x).cuda() for x in (off.view(np.int64), ln.view(np.int32), out, status))
        ctx.after_torch_stream(gd.device)
        st = _decode_icf(g4, master, batch, icf, G4_MEM_DEVICE, batch.arena.data_ptr(), int(batch.total_bytes), od.data_ptr(), ld.data_ptr(),
                         gd.data_ptr(), sd.data_ptr())
        ctx.synchronize()
        out, status = gd.cpu().numpy(), sd.cpu().numpy()
    else:
        a = np.ascontiguousarray(batch.arena)
        st = _decode_icf(g4, master, batch, icf, G4_MEM_HOST, a.ctypes.data, int(batch.total_bytes), off.ctypes.data, ln.ctypes.data,
                         out.ctypes.data, status.ctypes.data)
    assert st == G4_ERR_FORMAT
    assert status[7] == G4_ERR_FORMAT and (np.delete(status, 7) == G4_OK).all()
    for t in range(12):
        if t != 7:
            r, c = divmod(t, 4)
            blk = np.s_[r * 90:(r + 1) * 90, c * 120:(c + 1) * 120]
            assert np.array_equal(out[blk].view(np.uint32), want[blk].view(np.uint32)), t

    if device:  # asynchronous mode: the call only enqueues; status is read after synchronising
        ctx.set_async(True)
        try:
            gd = torch.empty((270, 480), dtype=torch.float32, device="cuda")
            sd = torch.full((12,), 99, dtype=torch.int32, device="cuda")
            ctx.after_torch_stream(gd.device)
            st = _decode_icf(g4, master, batch, icf, G4_MEM_DEVICE, batch.arena.data_ptr(), int(batch.arena.numel()), batch.offsets.data_ptr(),
                             batch.lens.data_ptr(), gd.data_ptr(), sd.data_ptr())
            assert st == G4_OK
            ctx.synchronize()
            assert not sd.cpu().numpy().any()
            assert np.array_equal(gd.cpu().numpy().view(np.uint32), want.view(np.uint32))
        finally:
            ctx.set_async(False)


@pytest.mark.gpu
def test_element_type_gating(g4):
    """Element type 3 keeps the status every existing entry point gave it; the ICF calls check their descriptor and band."""
    from gridfour_b200 import _lib

    L = _lib.lib()
    ctx = g4.Context.default()
    cl = g4.CodecSpecification().native_list()
    band = _lib.BandDesc(G4_ELEM_ICF, 4, 4, 1, 1, 4, 0, 0)
    grid = np.zeros((4, 4), np.float32)
    arena = np.zeros(256, np.uint8)
    off, ln = np.zeros(1, np.uint64), np.zeros(1, np.uint32)
    cod, pred, st = np.zeros(1, np.uint8), np.zeros(1, np.uint8), np.zeros(1, np.int32)
    total = C.c_uint64(0)
    assert L.g4_encode_tiles(ctx._h, C.byref(cl), C.byref(band), G4_MEM_HOST, grid.ctypes.data, arena.ctypes.data, 256, off.ctypes.data,
                             ln.ctypes.data, cod.ctypes.data, pred.ctypes.data, st.ctypes.data, C.byref(total)) == G4_ERR_ARG
    assert L.g4_decode_tiles(ctx._h, C.byref(cl), C.byref(band), G4_MEM_HOST, arena.ctypes.data, off.ctypes.data, ln.ctypes.data,
                             grid.ctypes.data, st.ctypes.data) == G4_ERR_ARG
    assert L.g4_decode_tiles_bounded(ctx._h, C.byref(cl), C.byref(band), G4_MEM_HOST, arena.ctypes.data, 256, off.ctypes.data,
                                     ln.ctypes.data, grid.ctypes.data, st.ctypes.data) == G4_ERR_ARG
    refs = (_lib.TileRef * 1)()
    refs[0].offset, refs[0].pitch = 0, 4
    assert L.g4_encode_tile_list(ctx._h, C.byref(cl), G4_ELEM_ICF, 4, 4, 1, G4_MEM_HOST, grid.ctypes.data, refs, arena.ctypes.data, 256,
                                 off.ctypes.data, ln.ctypes.data, cod.ctypes.data, pred.ctypes.data, st.ctypes.data,
                                 C.byref(total)) == G4_ERR_ARG
    assert L.g4_decode_tile_list(ctx._h, C.byref(cl), G4_ELEM_ICF, 4, 4, 1, G4_MEM_HOST, arena.ctypes.data, 256, off.ctypes.data,
                                 ln.ctypes.data, grid.ctypes.data, refs, st.ctypes.data) == G4_ERR_ARG
    d = _lib.IcfDesc(10.0, 0.0, INT_MIN, float("nan"))
    bad = _lib.IcfDesc(0.0, 0.0, INT_MIN, float("nan"))
    i32 = _lib.BandDesc(G4_ELEM_I32, 4, 4, 1, 1, 4, 0, 0)
    for b, desc in [(band, None), (band, bad), (i32, d)]:
        assert L.g4_encode_tiles_icf(ctx._h, C.byref(cl), C.byref(b), C.byref(desc) if desc else None, G4_MEM_HOST, grid.ctypes.data,
                                     arena.ctypes.data, 256, off.ctypes.data, ln.ctypes.data, cod.ctypes.data, pred.ctypes.data,
                                     st.ctypes.data, C.byref(total)) == G4_ERR_ARG
        assert L.g4_decode_tiles_icf(ctx._h, C.byref(cl), C.byref(b), C.byref(desc) if desc else None, G4_MEM_HOST, arena.ctypes.data,
                                     256, off.ctypes.data, ln.ctypes.data, grid.ctypes.data, st.ctypes.data) == G4_ERR_ARG
    # the descriptor does not outlive its call: type 3 is refused again afterwards
    assert L.g4_encode_tiles_icf(ctx._h, C.byref(cl), C.byref(band), C.byref(d), G4_MEM_HOST, grid.ctypes.data, arena.ctypes.data, 256,
                                 off.ctypes.data, ln.ctypes.data, cod.ctypes.data, pred.ctypes.data, st.ctypes.data, C.byref(total)) == G4_OK
    assert L.g4_decode_tiles(ctx._h, C.byref(cl), C.byref(band), G4_MEM_HOST, arena.ctypes.data, off.ctypes.data, ln.ctypes.data,
                             grid.ctypes.data, st.ctypes.data) == G4_ERR_ARG


@pytest.mark.gpu
def test_icf_sample_files(g4, oracle, icf_ref):
    import math

    from gridfour_b200 import gvrs

    files = sample_files()
    for name in ["Sample03_ICFNoComp.gvrs", "Sample07_ICFComp.gvrs", "Sample12_ICFNoComp.gvrs"]:
        img = gvrs.GvrsImage.parse(files[name])
        s = img.spec
        master = _master(g4, s.codecs) if s.codecs else g4.CodecMaster()
        got = img.read_raster(master, crop=True, as_float=True)
        r, c = np.mgrid[0:s.n_rows, 0:s.n_cols]
        assert got.dtype == np.float32 and np.array_equal(got, (r * s.n_cols + c - 1).astype(np.float32)), name
        codes = img.read_raster(master, crop=True)
        assert codes.dtype == np.int32 and np.array_equal(codes, r * s.n_cols + c - 1), name
        if name.startswith("Sample12"):
            full = img.read_raster(master, as_float=True)
            assert full.shape == (12, 12) and np.isnan(full[10:, :]).all() and np.isnan(full[:, 10:]).all()
    img = gvrs.GvrsImage.parse(files["Sample14_LSOP.gvrs"])
    master = _master(g4, ["LSOP12"])
    got = img.read_raster(master, as_float=True)
    off, lens, _st = img.locate_payloads(master._context(), 0)
    payload = img.image[int(off[0]):int(off[0]) + int(lens[0])]
    want = icf_ref.icf_to_float(oracle.master_decode_i32([ORACLE_IDS["LSOP12"]], 101, 101, payload), 1000.0, 0.0)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    exact = np.array([[math.sin(c / 100.0 * math.pi) * math.sin(r / 100.0 * math.pi) for c in range(101)] for r in range(101)])
    assert np.abs(got - exact).max() <= 0.0005 + 1e-7
    assert img.read_raster(master).dtype == np.int32


@pytest.fixture(scope="module")
def icf_file(g4, oracle, icf_ref):
    from gridfour_b200 import gvrs

    rows, cols = 500, 700
    f = oracle.terrain_f32(0, 0, rows, cols) / np.float32(100)
    f[100:130, 200:260] = np.nan
    f[400, :] = np.nan
    e = gvrs.ElementSpec.int_coded_float("z", 1000.0, -0.5)
    spec = gvrs.GvrsSpec(rows, cols, 90, 120, [e], ["GvrsHuffman", "GvrsDeflate", "LSOP12"], checksum=True)
    master = _master(g4, spec.codecs)
    w = gvrs.GvrsWriter(spec, uuid=bytes(range(16)), time_modified=1700000000000)
    for name, rid, typ, content, desc in gvrs.codec_metadata(spec.codecs):
        w.add_metadata(name, rid, typ, content, desc)
    batch = w.add_raster(master, f)
    return w.finish(master._context()), f, batch, master, spec


@pytest.mark.gpu
def test_writer_round_trip(g4, oracle, icf_ref, icf_file):
    from gridfour_b200 import gvrs

    image, f, batch, master, spec = icf_file
    img = gvrs.GvrsImage.parse(image)
    assert img.verify_checksums(master._context()) == len(img.records) + 1
    got = img.read_raster(master, crop=True, as_float=True)
    want = icf_ref.icf_to_float(icf_ref.icf_to_int(f, 1000.0, -0.5), 1000.0, -0.5)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # every payload is the oracle's packing of the mapped codes (the margin holds the fill code)
    full = np.full((6 * 90, 6 * 120), INT_MIN, np.int32)
    full[:500, :700] = icf_ref.icf_to_int(f, 1000.0, -0.5)
    ids = [ORACLE_IDS[c] for c in spec.codecs]
    off, lens, _st = img.locate_payloads(master._context(), 0)
    for t in range(36):
        r, c = divmod(t, 6)
        want_p = oracle.master_encode_i32(ids, np.ascontiguousarray(full[r * 90:(r + 1) * 90, c * 120:(c + 1) * 120]))
        assert batch.payload(t) == want_p, t
        assert img.image[int(off[t]):int(off[t]) + int(lens[t])] == want_p, t


@pytest.mark.gpu
def test_three_element_round_trip_and_device_read(g4, oracle, icf_ref):
    import torch

    from gridfour_b200 import gvrs

    rows, cols = 300, 400
    z = oracle.terrain_i32(0, 0, rows, cols)
    v = oracle.terrain_f32(700, 100, rows, cols)
    v[50:60, 70:300] = np.nan
    f = oracle.terrain_f32(900, 900, rows, cols)
    elements = [gvrs.ElementSpec.integer("z"), gvrs.ElementSpec.int_coded_float("v", 10.0, 0.0, -20000.0, 20000.0),
                gvrs.ElementSpec.floating("f")]
    codecs = ["GvrsHuffman", "GvrsDeflate", "GvrsFloat", "LSOP12"]
    spec = gvrs.GvrsSpec(rows, cols, 90, 120, elements, codecs, checksum=True)
    master = _master(g4, codecs)
    w = gvrs.GvrsWriter(spec, uuid=bytes(range(16)), time_modified=1700000000000)
    batches = w.add_rasters(master, [z, v, f])
    img = gvrs.GvrsImage.parse(w.finish(master._context()))
    got = img.read_rasters(master, crop=True, as_float=True)
    want_v = icf_ref.icf_to_float(icf_ref.icf_to_int(v, 10.0, 0.0), 10.0, 0.0)
    assert np.array_equal(got[0], z) and np.array_equal(got[2].view(np.uint32), f.view(np.uint32))
    assert got[1].dtype == np.float32 and np.array_equal(got[1].view(np.uint32), want_v.view(np.uint32))
    assert np.array_equal(img.read_rasters(master, crop=True)[1], icf_ref.icf_to_int(v, 10.0, 0.0))
    # device-resident read of the ICF element equals the host read
    host = img.read_raster(master, element=1, as_float=True)
    n = spec.tiles_down * spec.tiles_across
    pos = np.zeros(n, np.int64)
    for t, p in img.tile_directory().items():
        pos[t] = p
    dimg = torch.frombuffer(bytearray(img.image), dtype=torch.uint8).cuda()
    off, lens, st = gvrs.unpack_tile_records_multi_device(master._context(), dimg, torch.from_numpy(pos).cuda(), 3, True)
    torch.cuda.synchronize()
    assert int((st != 0).sum()) == 0
    band = master._band((spec.tiles_down * 90, spec.tiles_across * 120), np.float32, 90, 120)
    band.elem_type = G4_ELEM_ICF
    out = master.decodeTiles(g4.TileBatch(dimg, off[1], lens[1], None, None, None, int(dimg.numel()), band, elements[1].icf))
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint32), host.view(np.uint32))
    assert batches[1].icf == elements[1].icf


@pytest.mark.gpu
def test_tile_cache_float_accessors(g4, oracle, icf_ref, icf_file):
    from gridfour_b200 import gvrs

    image, f, _batch, master, spec = icf_file
    img = gvrs.GvrsImage.parse(image)
    whole = img.read_raster(master, as_float=True)
    cache = g4.RasterTileCache(img, master, max_tiles=8)
    blk = cache.readBlockFloat(70, 100, 40, 150)   # crosses two tile rows and two tile columns
    assert blk.dtype == np.float32 and np.array_equal(blk.view(np.uint32), whole[70:110, 100:250].view(np.uint32))
    assert cache.readValueFloat(95, 130).tobytes() == whole[95, 130].tobytes()
    assert np.array_equal(cache.readBlock(70, 100, 40, 150), icf_ref.icf_to_int(whole[70:110, 100:250], 1000.0, -0.5))
    rng = np.random.default_rng(3)
    new = rng.uniform(-30, 30, (20, 50)).astype(np.float32)
    new[3, 4] = np.nan
    cache.writeBlockFloat(80, 110, new)
    tiles, batch = cache.flush()
    assert tiles == [0, 1, 6, 7]
    decoded = master.decodeTiles(batch)   # the codes of the four tiles side by side, in list order
    codes = icf_ref.icf_to_int(new, 1000.0, -0.5)
    assert np.array_equal(decoded[80:90, 110:120], codes[:10, :10])
    assert np.array_equal(decoded[80:90, 120:160], codes[:10, 10:])
    assert np.array_equal(decoded[0:10, 240 + 110:240 + 120], codes[10:, :10])
    assert np.array_equal(decoded[0:10, 360:400], codes[10:, 10:])
    assert np.array_equal(cache.readBlockFloat(80, 110, 20, 50).view(np.uint32),
                          icf_ref.icf_to_float(codes, 1000.0, -0.5).view(np.uint32))
    with pytest.raises(ValueError):
        g4.RasterTileCache(gvrs.GvrsImage.parse(sample_files()["Sample05_IntComp.gvrs"]), g4.CodecMaster()).readBlockFloat(0, 0, 1, 1)
