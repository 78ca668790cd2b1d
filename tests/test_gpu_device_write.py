"""Writes from CUDA tensors (GvrsWriter.add_raster / add_rasters with tensors, CodecMaster.encodeTiles(padValue=...),
g4_encode_window): the edge tiles are padded on the device, and every result equals the host path on the same values padded
on the host, byte for byte."""
import ctypes as C
import struct

import numpy as np
import pytest

G4_OK, G4_ERR_ARG, G4_ERR_UNSUPPORTED = 0, -1, -5
G4_ELEM_I32, G4_ELEM_F32, G4_ELEM_I16, G4_ELEM_ICF = 0, 1, 2, 3

TR, TC = 20, 22          # tile size: the tile columns are not a multiple of 4, so tile edges fall at every residue
ROWS, COLS = 95, 127     # 5 x 6 tiles, the last row and column of tiles partial
UUID, TIME = bytes(range(16)), 1700000000000


@pytest.fixture(scope="module")
def g4():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gridfour_b200

    return gridfour_b200


def _master(g4, codecs, value_checksum=False, deflate=True):
    spec = g4.CodecSpecification(default=False)
    classes = {"GvrsHuffman": (g4.CodecHuffman,), "GvrsDeflate": (g4.CodecDeflate,), "GvrsFloat": (g4.CodecFloat,),
               "GvrsCanonicalHuffman": (g4.CodecCanonHuffman,), "LSOP12": (g4.LsEncoder12, g4.LsDecoder12)}
    for c in codecs:
        spec.addCompressionCodec(c, *classes[c])
    m = g4.CodecMaster(spec)
    if "LSOP12" in codecs:
        m.getEncoder("LSOP12").setValueChecksumEnabled(value_checksum)
        m.getEncoder("LSOP12").setDeflateEnabled(deflate)
    return m


def _cuda(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _bytes(a):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    return np.ascontiguousarray(a).view(np.uint8)


def _short_spec(name, fill):
    from gridfour_b200 import gvrs

    return gvrs.ElementSpec(gvrs.ELEM_SHORT, name, range_block=struct.pack("<hhh", -32767, 32767, fill))


def _grids(oracle, kinds, rows=ROWS, cols=COLS):
    out = []
    for k, kind in enumerate(kinds):
        if kind == "int":
            out.append(oracle.terrain_i32(100 * k, 300, rows, cols))
        elif kind == "float":
            out.append(oracle.terrain_f32(200 + k, 50, rows, cols))
        elif kind == "short":
            s = np.clip(oracle.terrain_i32(500, 100 * k, rows, cols) // 8, -30000, 30000).astype(np.int16)
            s[30:45, 40:70] = -9999     # the fill value: coded as null
            s[50:52, 10:20] = -32768    # not the fill value: stays a value
            out.append(s)
        else:  # integer-coded float values, with NaN (the fill) in a patch
            v = (oracle.terrain_f32(10, 20 + k, rows, cols) * np.float32(0.25)).astype(np.float32)
            v[60:70, 5:50] = np.nan
            out.append(v)
    return out


def _elements(kinds):
    from gridfour_b200 import gvrs

    make = {"int": lambda k: gvrs.ElementSpec.integer("e%d" % k, fill_value=-777),
            "float": lambda k: gvrs.ElementSpec.floating("e%d" % k, fill_value=-1.5),
            "short": lambda k: _short_spec("e%d" % k, -9999),
            "icf": lambda k: gvrs.ElementSpec.int_coded_float("e%d" % k, 100.0, 0.5)}
    return [make[kind](k) for k, kind in enumerate(kinds)]


CASES = {
    "int": (["int"], ["GvrsHuffman", "GvrsDeflate", "LSOP12"]),
    "float": (["float"], ["GvrsFloat"]),
    "short": (["short"], ["GvrsHuffman", "GvrsDeflate"]),
    "icf": (["icf"], ["GvrsHuffman", "GvrsDeflate", "LSOP12"]),
    "icf_codes": (["icf"], ["GvrsHuffman", "GvrsDeflate", "LSOP12"]),
    "three": (["float", "short", "icf"], ["GvrsHuffman", "GvrsDeflate", "GvrsFloat", "LSOP12"]),
}


def _case_grids(oracle, case):
    kinds, _ = CASES[case]
    grids = _grids(oracle, kinds)
    if case == "icf_codes":
        grids = [_elements(kinds)[0].icf.to_int(grids[0])]
    return grids


def _write(master, spec, grids):
    from gridfour_b200 import gvrs

    w = gvrs.GvrsWriter(spec, uuid=UUID, time_modified=TIME)
    for name, rid, typ, content, desc in gvrs.codec_metadata(spec.codecs):
        w.add_metadata(name, rid, typ, content, desc)
    batches = w.add_raster(master, grids[0]) if len(grids) == 1 else w.add_rasters(master, grids)
    return w.finish(master._context()), batches


@pytest.mark.gpu
@pytest.mark.parametrize("checksum", [True, False])
@pytest.mark.parametrize("case", list(CASES))
def test_device_written_image_equals_the_host_image(g4, oracle, case, checksum):
    from gridfour_b200 import gvrs

    kinds, codecs = CASES[case]
    master = _master(g4, codecs, value_checksum=checksum)
    spec = gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(kinds), codecs, checksum=checksum)
    grids = _case_grids(oracle, case)
    host, _ = _write(master, spec, grids)
    dev, batches = _write(master, spec, [_cuda(g) for g in grids])
    assert dev == host, case
    for b in batches if isinstance(batches, list) else [batches]:
        assert b.arena.is_cuda and b.offsets.is_cuda and b.lens.is_cuda
    # the image reads back as the source raster, bit for bit; ICF values as the host writer's file reads back
    img = gvrs.GvrsImage.parse(dev)
    assert img.verify_checksums(master._context()) == (len(img.records) + 1 if checksum else 0)
    dimg = img.to_device()
    for k, (e, g) in enumerate(zip(spec.elements, grids)):
        got = dimg.read_raster(master, element=k, crop=True)
        if e.type_code == gvrs.ELEM_INT_CODED_FLOAT and g.dtype == np.float32:
            want = gvrs.GvrsImage.parse(host).read_raster(master, element=k, crop=True, as_float=True)
            assert np.array_equal(_bytes(dimg.read_raster(master, element=k, crop=True, as_float=True)), _bytes(want))
            assert np.array_equal(_bytes(got), _bytes(e.icf.to_int(g)))
        elif e.type_code == gvrs.ELEM_SHORT:   # the fill value reads back as SHORT_NULL_CODE (TileElementShort.decode)
            assert np.array_equal(_bytes(got), _bytes(np.where(g == e.fill_value, np.int16(-32768), g))), (case, k)
        else:
            assert np.array_equal(_bytes(got), _bytes(g)), (case, k)


# ---- g4_encode_window against g4_encode_tiles(_icf) on a copy padded with torch ---------------------------------------------
def _padded(t, pad, tr, tc):
    import torch

    rows, cols = t.shape
    full = torch.full((-(-rows // tr) * tr, -(-cols // tc) * tc), pad, dtype=t.dtype, device=t.device)
    full[:rows, :cols] = t
    return full


def _same_batch(a, b):
    assert a.total_bytes == b.total_bytes
    assert np.array_equal(_bytes(a.arena[:a.total_bytes]), _bytes(b.arena[:b.total_bytes]))
    for x, y in [(a.offsets, b.offsets), (a.lens, b.lens), (a.codec, b.codec), (a.predictor, b.predictor), (a.status, b.status)]:
        assert np.array_equal(_bytes(x), _bytes(y))


RAW_ROWS, RAW_COLS = 99, 131   # 5 x 6 tiles again, but the edge tiles hold a single row or column of margin


def _noisy_edges(a, rng):
    """Full-range noise in the cells next to the margin.  Noise costs more than 4 bytes per int (2 per short) in every
    codec, and the margin of an edge tile is only 1 row or column wide, so the edge tiles of int and short rasters are
    stored raw."""
    a = a.copy()
    info = np.iinfo(a.dtype) if a.dtype.kind == "i" else None
    r0, c0 = (a.shape[0] // TR) * TR, (a.shape[1] // TC) * TC
    for sl in [(slice(r0, None), slice(None)), (slice(None), slice(c0, None))]:
        shape = a[sl].shape
        if info is not None:
            a[sl] = rng.integers(info.min + 1, info.max, size=shape, dtype=np.int64).astype(a.dtype)
        else:
            a[sl] = rng.integers(0, 2 ** 32, size=shape, dtype=np.uint64).astype(np.uint32).view(np.float32)
    return a


def _parity_cases(oracle):
    from gridfour_b200 import IntCodedFloat

    rng = np.random.default_rng(7)
    ints, floats, shorts, values = _grids(oracle, ["int", "float", "short", "icf"])
    r_ints, r_floats, r_shorts, r_values = [_noisy_edges(g, rng) for g in _grids(oracle, ["int", "float", "short", "icf"], RAW_ROWS, RAW_COLS)]
    huff = ["GvrsHuffman", "GvrsDeflate"]
    lsop = ["GvrsHuffman", "GvrsDeflate", "LSOP12"]
    nan_icf = IntCodedFloat(100.0, 0.5)
    finite_icf = IntCodedFloat(10.0, -3.0, fill_int=-4000000, fill_value=-250.0)
    return [
        # (name, master args, grid, fillValue, icf, padValue)
        ("int", (lsop,), ints, None, None, -777),
        ("int_raw_edges", (huff,), r_ints, None, None, 0),
        ("float_nan", (["GvrsFloat"],), floats, None, None, float("nan")),
        ("float_neg", (["GvrsFloat"],), floats, None, None, -1.5),
        ("float_noisy_edges", (["GvrsFloat"],), r_floats, None, None, -1.5),
        ("short_fill_is_pad", (huff,), shorts, -9999, None, -9999),                 # -9999 null inside and in the margin
        ("short_other_pad", (huff,), shorts, -9999, None, -32768),                 # -32768 stays a value everywhere
        ("short_raw_edges", (huff,), r_shorts, -9999, None, -9999),
        ("short_lsop", (lsop,), shorts, -9999, None, -9999),
        ("icf_nan", (lsop,), values, None, nan_icf, float("nan")),
        ("icf_finite_fill", (lsop,), values, None, finite_icf, -250.0),
        ("icf_noisy_edges", (huff,), r_values, None, nan_icf, float("nan")),
        ("lsop_value_checksum", (["LSOP12"], True, True), ints, None, None, -777),
        ("lsop_no_deflate", (["LSOP12"], False, False), ints, None, None, -777),
        ("lsop_both", (["LSOP12"], True, False), shorts, -9999, None, -9999),
    ]


@pytest.mark.gpu
def test_encode_window_equals_encode_tiles_on_a_padded_copy(g4, oracle):
    for name, margs, grid, fill, icf, pad in _parity_cases(oracle):
        master = _master(g4, *margs)
        t = _cuda(grid)
        got = master.encodeTiles(t, TR, TC, fillValue=fill, icf=icf, padValue=pad)
        want = master.encodeTiles(_padded(t, pad, TR, TC), TR, TC, fillValue=fill, icf=icf)
        try:
            _same_batch(got, want)
        except AssertionError as e:
            raise AssertionError(name) from e
        assert got.band.tiles_down == 5 and got.band.tiles_across == 6
        if "raw_edges" in name:   # the edge tiles other than the corner (whose margin is larger) are stored raw
            codec = got.codec.cpu().numpy().reshape(5, 6)
            assert (codec[-1, :-1] == 255).all() and (codec[:-1, -1] == 255).all(), (name, codec)


@pytest.mark.gpu
def test_encode_window_large_partial_tiles_through_lsop12(g4, oracle):
    master = _master(g4, ["LSOP12"], value_checksum=True)
    grid = _cuda(oracle.terrain_i32(40, 70, 1100, 1300))
    got = master.encodeTiles(grid, 512, 512, padValue=-(2 ** 31))
    want = master.encodeTiles(_padded(grid, -(2 ** 31), 512, 512), 512, 512)
    _same_batch(got, want)
    assert got.band.tiles_down == 3 and got.band.tiles_across == 3
    assert np.array_equal(_bytes(master.decodeTiles(got)[:1100, :1300]), _bytes(grid))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["int", "short", "icf"])
def test_pitched_sources(g4, oracle, kind):
    """A slice of a wider tensor: start column and pitch at every residue mod 4 (16-byte and scalar paths)."""
    import torch

    from gridfour_b200 import IntCodedFloat

    grid = _grids(oracle, [kind])[0]
    master = _master(g4, ["GvrsHuffman", "GvrsDeflate", "LSOP12"])
    icf = IntCodedFloat(100.0, 0.5) if kind == "icf" else None
    fill = -9999 if kind == "short" else None
    pad = {"int": -777, "short": -9999, "icf": float("nan")}[kind]
    want = master.encodeTiles(_cuda(grid), TR, TC, fillValue=fill, icf=icf, padValue=pad)
    for col0 in range(4):
        for extra in range(4):
            wide = torch.full((ROWS, COLS + 4 + extra), 3, dtype=_cuda(grid).dtype, device="cuda")
            view = wide[:, col0:col0 + COLS]
            view.copy_(_cuda(grid))
            assert view.stride(0) % 4 == (COLS + extra) % 4
            got = master.encodeTiles(view, TR, TC, fillValue=fill, icf=icf, padValue=pad)
            _same_batch(got, want)


@pytest.mark.gpu
def test_launch_counts(g4, oracle):
    from gridfour_b200 import IntCodedFloat

    ints, floats, shorts, values = _grids(oracle, ["int", "float", "short", "icf"])
    aligned_rows, aligned_cols = 4 * TR, 5 * TC
    for grid, codecs, pad in [(ints, ["GvrsHuffman", "GvrsDeflate", "LSOP12"], -777), (floats, ["GvrsFloat"], -1.5)]:
        master = _master(g4, codecs)
        ctx = master._context()
        # tile-aligned: straight from the tensor, the launches of g4_encode_tiles and the same results
        t = _cuda(grid[:aligned_rows, :aligned_cols])
        n0 = ctx.launch_count
        got = master.encodeTiles(t, TR, TC, padValue=pad)
        n1 = ctx.launch_count
        want = master.encodeTiles(t, TR, TC)
        n2 = ctx.launch_count
        assert n1 - n0 == n2 - n1
        _same_batch(got, want)
        # unaligned: one load pass more
        t = _cuda(grid)
        p = _padded(t, pad, TR, TC)
        n0 = ctx.launch_count
        master.encodeTiles(t, TR, TC, padValue=pad)
        n1 = ctx.launch_count
        master.encodeTiles(p, TR, TC)
        n2 = ctx.launch_count
        assert n1 - n0 == n2 - n1 + 1
    # short and ICF: the load pass stands in for the widening / mapping launch
    for grid, fill, icf, pad in [(shorts, -9999, None, -9999), (values, None, IntCodedFloat(100.0, 0.5), float("nan"))]:
        master = _master(g4, ["GvrsHuffman", "GvrsDeflate", "LSOP12"])
        ctx = master._context()
        t = _cuda(grid)
        p = _padded(t, pad, TR, TC)
        n0 = ctx.launch_count
        master.encodeTiles(t, TR, TC, fillValue=fill, icf=icf, padValue=pad)
        n1 = ctx.launch_count
        master.encodeTiles(p, TR, TC, fillValue=fill, icf=icf)
        n2 = ctx.launch_count
        assert n1 - n0 == n2 - n1


@pytest.mark.gpu
def test_c_call_rejects_bad_arguments(g4, oracle):
    import torch

    from gridfour_b200 import IntCodedFloat, _lib

    L = _lib.lib()
    master = _master(g4, ["GvrsHuffman", "GvrsDeflate"])
    ctx = master._context()
    src = _cuda(_grids(oracle, ["float"])[0])
    nT = 30
    arena = torch.empty(nT * 4 * TR * TC + 64, dtype=torch.uint8, device="cuda")
    offsets = torch.empty(nT, dtype=torch.int64, device="cuda")
    lens, status = torch.empty(nT, dtype=torch.int32, device="cuda"), torch.empty(nT, dtype=torch.int32, device="cuda")
    codec, pred = torch.empty(nT, dtype=torch.uint8, device="cuda"), torch.empty(nT, dtype=torch.uint8, device="cuda")
    icf = IntCodedFloat(100.0, 0.5).desc()
    bad_icf = _lib.IcfDesc()
    bad_icf.scale = float("inf")
    total = C.c_uint64(0)

    def band(elem=G4_ELEM_ICF, down=5, across=6, tr=TR, tc=TC):
        b = _lib.BandDesc()
        b.elem_type, b.tile_rows, b.tile_cols, b.tiles_down, b.tiles_across = elem, tr, tc, down, across
        b.grid_pitch = across * tc
        return b

    def call(b, d, n_rows=ROWS, n_cols=COLS, pitch=COLS):
        return L.g4_encode_window(ctx._h, C.byref(master._native_list()), C.byref(b), None if d is None else C.byref(d), n_rows, n_cols,
                                  src.data_ptr(), pitch, 0x7fc00000, arena.data_ptr(), int(arena.numel()), offsets.data_ptr(),
                                  lens.data_ptr(), codec.data_ptr(), pred.data_ptr(), status.data_ptr(), C.byref(total))

    assert call(band(), icf) == G4_OK
    assert call(band(G4_ELEM_I32), None) == G4_OK                                       # the bits as int32 codes
    assert call(band(G4_ELEM_F32), None) == G4_OK
    for args in [(band(), icf, 0, COLS), (band(), icf, ROWS, 0),                         # empty
                 (band(down=4), icf), (band(down=6), icf), (band(across=5), icf), (band(across=7), icf),  # tile counts
                 (band(), icf, ROWS, COLS, COLS - 1),                                    # src_pitch < n_cols
                 (band(7), None), (band(down=0), icf, 0, COLS),                          # bad raster
                 (band(G4_ELEM_I32), icf), (band(G4_ELEM_I16), icf),                     # a descriptor for a non-ICF element
                 (band(), bad_icf), (band(), None)]:                                     # an invalid descriptor, none for ICF
        assert call(*args) == G4_ERR_ARG, args
    assert call(band(G4_ELEM_F32, down=95, tr=1), None) == G4_ERR_UNSUPPORTED


@pytest.mark.gpu
def test_python_rejections(g4, oracle):
    import torch

    from gridfour_b200 import gvrs

    kinds, codecs = CASES["three"]
    master = _master(g4, codecs)
    spec = gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(kinds), codecs, checksum=True)
    grids = _grids(oracle, kinds)
    tensors = [_cuda(g) for g in grids]
    w = gvrs.GvrsWriter(spec)
    with pytest.raises(ValueError):   # numpy arrays and tensors mixed
        w.add_rasters(master, [grids[0], tensors[1], tensors[2]])
    with pytest.raises(ValueError):   # a wrong dtype (the short element as int32)
        w.add_rasters(master, [tensors[0], tensors[1].to(torch.int32), tensors[2]])
    with pytest.raises(ValueError):   # a wrong shape
        w.add_rasters(master, [tensors[0], tensors[1], tensors[2][:-1]])
    with pytest.raises(ValueError):   # a tensor that is not on the GPU
        w.add_rasters(master, [tensors[0], tensors[1].cpu(), tensors[2]])
    one = gvrs.GvrsWriter(gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(["int"]), codecs))
    t = _cuda(_grids(oracle, ["int"])[0])
    for bad in [t[:, :-1], t.to(torch.int64), t.to(torch.float32), t.cpu()]:
        with pytest.raises(ValueError):
            one.add_raster(master, bad)
    wide = torch.zeros((ROWS, 2 * COLS), dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError):   # rows not contiguous
        one.add_raster(master, wide[:, ::2])
    with pytest.raises(ValueError):   # padValue is for CUDA tensors only
        master.encodeTiles(grids[0], TR, TC, padValue=0.0)
    assert len(one.buf) == one.header_size + gvrs.FILEPOS_HEADER_RECORD and not one.tile_positions   # nothing was written
    # a slice of a wider tensor (contiguous rows, any pitch) is accepted and writes the same file
    wide[:, 3:3 + COLS] = t
    a = gvrs.GvrsWriter(gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(["int"]), codecs), uuid=UUID)
    a.add_raster(master, wide[:, 3:3 + COLS])
    b = gvrs.GvrsWriter(gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(["int"]), codecs), uuid=UUID)
    b.add_raster(master, t.cpu().numpy())
    assert a.finish(master._context()) == b.finish(master._context())
