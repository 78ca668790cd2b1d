"""Reads from a GVRS file image resident on the GPU (GvrsImage.to_device, GvrsDeviceImage.read_block / read_raster,
g4_decode_window): every result equals the host read_raster, cropped with numpy, byte for byte."""
import ctypes as C
import struct
import warnings

import numpy as np
import pytest

from gvrs_common import sample_files

G4_OK, G4_DECLINED, G4_CHECKSUM_MISMATCH = 0, 1, 2
G4_ERR_ARG, G4_ERR_FORMAT = -1, -2
G4_ELEM_I32, G4_ELEM_F32, G4_ELEM_I16, G4_ELEM_ICF = 0, 1, 2, 3
G4_MEM_DEVICE = 1
INT_MIN = -(2 ** 31)


@pytest.fixture(scope="module")
def g4():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gridfour_b200

    return gridfour_b200


def _master(g4, codecs):
    spec = g4.CodecSpecification(default=False)
    classes = {"GvrsHuffman": (g4.CodecHuffman,), "GvrsDeflate": (g4.CodecDeflate,), "GvrsFloat": (g4.CodecFloat,),
               "GvrsCanonicalHuffman": (g4.CodecCanonHuffman,), "LSOP12": (g4.LsEncoder12, g4.LsDecoder12)}
    for c in codecs:
        spec.addCompressionCodec(c, *classes[c])
    return g4.CodecMaster(spec)


def _bytes(a):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    return np.ascontiguousarray(a).view(np.uint8)


def _float_modes(e):
    from gridfour_b200 import gvrs

    return (False, True) if e.type_code == gvrs.ELEM_INT_CODED_FLOAT else (False,)


@pytest.mark.gpu
def test_reference_files_read_as_the_host_reads_them(g4):
    from gridfour_b200 import gvrs

    n_files = 0
    for name, image in sample_files().items():
        img = gvrs.GvrsImage.parse(image)
        s = img.spec
        master = _master(g4, s.codecs)
        dimg = img.to_device()
        for k, e in enumerate(s.elements):
            for as_float in _float_modes(e):
                for crop in (False, True):
                    host = img.read_raster(master, element=k, crop=crop, as_float=as_float)
                    dev = dimg.read_raster(master, element=k, crop=crop, as_float=as_float)
                    assert dev.is_cuda and dev.shape == host.shape and str(dev.dtype).endswith(host.dtype.name), (name, k)
                    assert np.array_equal(_bytes(dev), _bytes(host)), (name, k, crop, as_float)
        n_files += 1
    assert n_files == 17


# ---- written images -----------------------------------------------------------------------------------------------------
TR, TC = 20, 22          # tile size: the tile columns are not a multiple of 4, so tile edges fall at every residue
ROWS, COLS = 95, 127     # 5 x 6 tiles, the last row and column of tiles partial
DROP = (1, 8, 29)        # tiles left out of the directory (29 is the partial corner tile)


def _short_spec(name, fill):
    from gridfour_b200 import gvrs

    return gvrs.ElementSpec(gvrs.ELEM_SHORT, name, range_block=struct.pack("<hhh", -32767, 32767, fill))


def _grids(oracle, kinds):
    out = []
    for k, kind in enumerate(kinds):
        if kind == "int":
            out.append(oracle.terrain_i32(100 * k, 300, ROWS, COLS))
        elif kind == "float":
            out.append(oracle.terrain_f32(200 + k, 50, ROWS, COLS))
        elif kind == "short":
            s = np.clip(oracle.terrain_i32(500, 100 * k, ROWS, COLS) // 8, -30000, 30000).astype(np.int16)
            s[30:45, 40:70] = -9999
            out.append(s)
        else:  # integer-coded float values, with NaN (the fill) in a patch
            v = (oracle.terrain_f32(10, 20 + k, ROWS, COLS) * np.float32(0.25)).astype(np.float32)
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


def _write(g4, master, spec, grids, drop=DROP):
    from gridfour_b200 import gvrs

    ctx = master._context()
    w = gvrs.GvrsWriter(spec, uuid=bytes(range(16)), time_modified=1700000000000)
    for name, rid, typ, content, desc in gvrs.codec_metadata(spec.codecs):
        w.add_metadata(name, rid, typ, content, desc)
    batches = [w._encode_element(master, e, g) for e, g in zip(spec.elements, grids)]
    keep = [t for t in range(spec.tiles_down * spec.tiles_across) if t not in drop]
    w.add_tile_records_multi(ctx, [b.arena for b in batches], [np.asarray(b.offsets)[keep] for b in batches],
                             [np.asarray(b.lens)[keep] for b in batches], tile_index=keep)
    return gvrs.GvrsImage.parse(w.finish(ctx))


CASES = {
    "int": (["int"], ["GvrsHuffman", "GvrsDeflate", "LSOP12"]),
    "float": (["float"], ["GvrsFloat"]),
    "short": (["short"], ["GvrsHuffman", "GvrsDeflate"]),
    "icf": (["icf"], ["GvrsHuffman", "GvrsDeflate", "LSOP12"]),
    "three": (["float", "short", "icf"], ["GvrsHuffman", "GvrsDeflate", "GvrsFloat", "LSOP12"]),
}


@pytest.fixture(scope="module")
def written(g4, oracle):
    from gridfour_b200 import gvrs

    out = {}
    for key, (kinds, codecs) in CASES.items():
        master = _master(g4, codecs)
        spec = gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(kinds), codecs, checksum=True)
        out[key] = (master, _write(g4, master, spec, _grids(oracle, kinds)))
    return out


def _windows():
    R, Cc = TR, TC
    w = []
    for r, c in [(0, 0), (R - 1, Cc - 1), (R, Cc), (R - 1, Cc), (R, Cc - 1), (2 * R - 1, 3 * Cc), (ROWS - 1, COLS - 1)]:
        w.append((r, c, 1, 1))                                            # single cells at tile corners
    w += [(R - 1, 0, 1, COLS), (ROWS - 1, 3, 1, COLS - 5), (0, Cc - 1, ROWS, 1), (5, COLS - 1, ROWS - 5, 1)]  # rows, columns
    for a in range(4):
        for b in range(4):
            w.append((R // 2 + a, Cc - 3 + a, R + 3, 2 * Cc - 5 + b))     # col0 and n_cols at every residue mod 4
    w += [(R, 2 * Cc, R, Cc), (0, Cc, R, Cc),                            # whole tiles (the second is absent)
          (R, Cc, 2 * R, 3 * Cc), (0, 0, 3 * R, 2 * Cc),                  # tile-aligned multi-tile blocks
          (ROWS - R - 3, COLS - Cc - 5, R + 3, Cc + 5), (4 * R, 5 * Cc, ROWS - 4 * R, COLS - 5 * Cc), (0, 0, ROWS, COLS)]
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_blocks_equal_the_host_raster(g4, written, case):
    import torch

    master, img = written[case]
    dimg = img.to_device()
    assert int((dimg.status == G4_DECLINED).sum()) == len(DROP)
    for k, e in enumerate(img.spec.elements):
        for as_float in _float_modes(e):
            host = img.read_raster(master, element=k, as_float=as_float)
            for (r, c, n, m) in _windows():
                want = host[r:r + n, c:c + m]
                got = dimg.read_block(master, r, c, n, m, element=k, as_float=as_float)
                assert got.shape == (n, m) and np.array_equal(_bytes(got), _bytes(want)), (case, k, as_float, (r, c, n, m))
                # into a strided slice of a larger mosaic: the margins stay as they were
                mosaic = torch.full((n + 7, m + 13), 0x5A, dtype=got.dtype, device=got.device)
                before = mosaic.clone()
                view = mosaic[3:3 + n, 5:5 + m]
                assert dimg.read_block(master, r, c, n, m, element=k, as_float=as_float, out=view) is view
                assert np.array_equal(_bytes(view), _bytes(want)), (case, k, as_float, (r, c, n, m))
                view.copy_(before[3:3 + n, 5:5 + m])
                assert np.array_equal(_bytes(mosaic), _bytes(before)), (case, k, as_float, (r, c, n, m))
            for crop in (False, True):
                want = img.read_raster(master, element=k, crop=crop, as_float=as_float)
                assert np.array_equal(_bytes(dimg.read_raster(master, element=k, crop=crop, as_float=as_float)), _bytes(want))


@pytest.mark.gpu
def test_absent_tiles_are_declined_not_errors(g4, written):
    master, img = written["int"]
    dimg = img.to_device()
    dimg.read_block(master, 0, 0, 2 * TR, 3 * TC)   # tiles 0, 1, 2, 6, 7, 8 of the raster; 1 and 8 are absent
    assert dimg.lastStatus.cpu().tolist() == [G4_OK, G4_DECLINED, G4_OK, G4_OK, G4_OK, G4_DECLINED]
    dimg.read_block(master, 3, 5, 2 * TR, 3 * TC)   # unaligned: tile rows 0..2, tile columns 0..3
    assert dimg.lastStatus.cpu().tolist() == [G4_OK, G4_DECLINED, G4_OK, G4_OK, G4_OK, G4_OK, G4_DECLINED, G4_OK] + [G4_OK] * 4


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["int", "float"])
def test_tile_aligned_reads_add_two_launches_to_the_band_decode(g4, written, case):
    import torch

    from gridfour_b200 import _lib

    master, img = written[case]
    dimg = img.to_device()
    ctx, spec = dimg.context, img.spec
    r0, c0, td, ta = 2, 1, 2, 3    # tiles 13..15 and 19..21: all present
    idx = torch.tensor([(r0 + i) * spec.tiles_across + c0 + j for i in range(td) for j in range(ta)], device=dimg.device)
    off = dimg.payload_off[0][idx].contiguous()
    lens = dimg.lens[0][idx].contiguous()
    band = _lib.BandDesc()
    band.elem_type = G4_ELEM_F32 if case == "float" else G4_ELEM_I32
    band.tile_rows, band.tile_cols, band.tiles_down, band.tiles_across, band.grid_pitch = TR, TC, td, ta, ta * TC
    grid = torch.empty((td * TR, ta * TC), dtype=torch.float32 if case == "float" else torch.int32, device=dimg.device)
    status = torch.empty(td * ta, dtype=torch.int32, device=dimg.device)
    n0 = ctx.launch_count
    got = dimg.read_block(master, r0 * TR, c0 * TC, td * TR, ta * TC)
    n1 = ctx.launch_count
    assert _lib.lib().g4_decode_tiles_bounded(ctx._h, C.byref(master._native_list()), C.byref(band), G4_MEM_DEVICE, dimg.image.data_ptr(),
                                              int(dimg.image.numel()), off.data_ptr(), lens.data_ptr(), grid.data_ptr(),
                                              status.data_ptr()) == G4_OK
    n2 = ctx.launch_count
    assert (n1 - n0) - (n2 - n1) == 2
    assert np.array_equal(_bytes(got), _bytes(grid))


def _payload_location(img, t, element=0):
    """File offset and length of element `element` of tile t, read off the record on the host."""
    pos = img.tile_directory()[t] + 4
    for _ in range(element):
        pos += 4 + struct.unpack_from("<i", img.image, pos)[0]
    return pos + 4, struct.unpack_from("<i", img.image, pos)[0]


@pytest.mark.gpu
def test_a_malformed_payload_fails_only_the_windows_that_touch_it(g4, oracle):
    from gridfour_b200 import gvrs

    codecs = ["GvrsHuffman", "GvrsDeflate", "LSOP12"]
    master = _master(g4, codecs)
    spec = gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(["int"]), codecs, checksum=False)
    img = _write(g4, master, spec, _grids(oracle, ["int"]), drop=())
    clean = img.read_raster(master)
    victim = 2 * spec.tiles_across + 3   # tile row 2, tile column 3
    off, ln = _payload_location(img, victim)
    assert ln < 4 * TR * TC              # a codec packing, not a raw tile
    bad = bytearray(img.image)
    bad[off] = 200                       # packing[0]: no codec has that index (CodecMaster.decode throws)
    dimg = gvrs.GvrsImage.parse(bytes(bad)).to_device()
    for (r, c, n, m) in _windows():
        touches = r // TR <= 2 <= (r + n - 1) // TR and c // TC <= 3 <= (c + m - 1) // TC
        if touches:
            with pytest.raises(g4.FormatError):
                dimg.read_block(master, r, c, n, m)
            st = dimg.lastStatus.cpu().numpy()
            ta = (c + m - 1) // TC - c // TC + 1
            assert st[(2 - r // TR) * ta + (3 - c // TC)] == G4_ERR_FORMAT and np.count_nonzero(st) == 1
        else:
            got = dimg.read_block(master, r, c, n, m)
            assert np.array_equal(_bytes(got), _bytes(clean[r:r + n, c:c + m])), (r, c, n, m)


@pytest.mark.gpu
def test_a_value_checksum_mismatch_warns_and_delivers(g4, oracle):
    from gridfour_b200 import gvrs

    master = _master(g4, ["LSOP12"])
    master.getEncoder("LSOP12").setValueChecksumEnabled(True)
    rows, cols, tr, tc = 180, 240, 60, 80
    grid = oracle.terrain_i32(900, 1200, rows, cols)
    spec = gvrs.GvrsSpec(rows, cols, tr, tc, [gvrs.ElementSpec.integer("z")], ["LSOP12"], checksum=False)
    img = _write(g4, master, spec, [grid], drop=())
    victim = None
    for t in range(9):
        off, ln = _payload_location(img, t)
        p = img.image[off:off + ln]
        if ln < 4 * tr * tc and p[1] & 0x80:
            victim = t
            break
    assert victim is not None
    bad = bytearray(img.image)
    bad[off + (55 if (p[1] & 0x0F) == 2 else 63)] ^= 0x10   # the stored CRC-32C of the values (LsHeader)
    dimg = gvrs.GvrsImage.parse(bytes(bad)).to_device()
    vr, vc = divmod(victim, 3)
    with pytest.warns(g4.ValueChecksumWarning):
        got = dimg.read_block(master, vr * tr + 5, vc * tc + 7, 30, 41)
    assert np.array_equal(got.cpu().numpy(), grid[vr * tr + 5:vr * tr + 35, vc * tc + 7:vc * tc + 48])
    assert dimg.lastStatus.cpu().tolist() == [G4_CHECKSUM_MISMATCH]
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        other = (victim + 1) % 9
        r, c = divmod(other, 3)
        assert np.array_equal(dimg.read_block(master, r * tr, c * tc, tr, tc).cpu().numpy(), grid[r * tr:(r + 1) * tr, c * tc:(c + 1) * tc])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["int", "three"])
def test_damaged_records_raise_in_to_device(g4, written, case):
    from gridfour_b200 import gvrs

    _, img = written[case]
    t = 4
    pos = img.tile_directory()[t]
    # a record that is not a tile record
    bad = bytearray(img.image)
    bad[pos - 4] = gvrs.RECORD_METADATA
    with pytest.raises(IOError):
        gvrs.GvrsImage.parse(bytes(bad)).to_device()
    # a payload byte flipped: the record checksum differs
    bad = bytearray(img.image)
    bad[pos + 12] ^= 0x01
    with pytest.raises(IOError):
        gvrs.GvrsImage.parse(bytes(bad)).to_device()
    gvrs.GvrsImage.parse(bytes(bad)).to_device(verify=False)   # not checked without verify


@pytest.mark.gpu
def test_async_reads_and_bad_windows(g4, written):
    import torch

    master, img = written["three"]
    dimg = img.to_device()
    ctx = dimg.context
    host = img.read_raster(master, element=2, as_float=True)
    ctx.set_async(True)
    try:
        outs = [dimg.read_block(master, r, c, n, m, element=2, as_float=True) for (r, c, n, m) in _windows()]
        statuses = [dimg.lastStatus]
        ctx.synchronize()
    finally:
        ctx.set_async(False)
    for (r, c, n, m), got in zip(_windows(), outs):
        assert np.array_equal(_bytes(got), _bytes(host[r:r + n, c:c + m])), (r, c, n, m)
    assert statuses[0].cpu().tolist() == [G4_DECLINED if t in DROP else G4_OK for t in range(30)]   # the last window: every tile
    for (r, c, n, m) in [(-1, 0, 1, 1), (0, -1, 1, 1), (0, 0, 0, 4), (0, 0, 4, 0), (ROWS - 1, 0, 2, 1), (0, COLS - 3, 1, 4)]:
        with pytest.raises(ValueError):
            dimg.read_block(master, r, c, n, m)
    with pytest.raises(ValueError):
        dimg.read_block(master, 0, 0, 1, 1, element=3)
    with pytest.raises(ValueError):   # rows not contiguous
        dimg.read_block(master, 0, 0, 4, 4, out=torch.empty((4, 8), dtype=torch.int32, device=dimg.device)[:, ::2])


@pytest.mark.gpu
def test_c_call_rejects_bad_arguments(g4, written):
    import torch

    from gridfour_b200 import _lib

    master, img = written["icf"]
    dimg = img.to_device()
    L, ctx = _lib.lib(), dimg.context
    spec = img.spec
    out = torch.empty((spec.tiles_down * TR, spec.tiles_across * TC), dtype=torch.float32, device=dimg.device)
    st = torch.empty(spec.tiles_down * spec.tiles_across, dtype=torch.int32, device=dimg.device)
    icf = spec.elements[0].icf.desc()
    bad_icf = _lib.IcfDesc()
    bad_icf.scale = 0.0

    def band(elem=G4_ELEM_ICF, down=spec.tiles_down):
        b = _lib.BandDesc()
        b.elem_type, b.tile_rows, b.tile_cols, b.tiles_down, b.tiles_across = elem, TR, TC, down, spec.tiles_across
        b.grid_pitch = spec.tiles_across * TC
        return b

    def call(b, d, row0, col0, n_rows, n_cols, pitch):
        return L.g4_decode_window(ctx._h, C.byref(master._native_list()), C.byref(b), None if d is None else C.byref(d), dimg.image.data_ptr(),
                                  int(dimg.image.numel()), dimg.payload_off[0].data_ptr(), dimg.lens[0].data_ptr(), dimg.status.data_ptr(),
                                  0, row0, col0, n_rows, n_cols, out.data_ptr(), pitch, st.data_ptr())

    R, Cc = spec.tiles_down * TR, spec.tiles_across * TC
    assert call(band(), icf, 3, 4, 10, 10, Cc) == G4_OK
    assert call(band(), icf, 0, 0, R, Cc, Cc) == G4_OK
    assert call(band(G4_ELEM_I32), None, 3, 4, 10, 10, Cc) == G4_OK                 # the codes
    for args in [(band(), icf, 0, 0, 0, 5, Cc), (band(), icf, 0, 0, 5, 0, Cc),       # empty
                 (band(), icf, -1, 0, 5, 5, Cc), (band(), icf, 0, -1, 5, 5, Cc),     # outside the tile grid
                 (band(), icf, R - 4, 0, 5, 5, Cc), (band(), icf, 0, Cc - 4, 5, 5, Cc),
                 (band(), icf, 0, 0, 5, 10, 9),                                      # out_pitch < n_cols
                 (band(7), None, 0, 0, 5, 5, Cc), (band(down=0), icf, 0, 0, 5, 5, Cc),  # bad raster
                 (band(G4_ELEM_I32), icf, 0, 0, 5, 5, Cc),                           # a descriptor for a non-ICF element
                 (band(), bad_icf, 0, 0, 5, 5, Cc), (band(), None, 0, 0, 5, 5, Cc)]:  # an invalid descriptor, none for ICF
        assert call(*args) == G4_ERR_ARG, args
