"""Point reads from a GVRS file image resident on the GPU (GvrsDeviceImage.read_values, g4_decode_points): every value equals
the host read_raster(crop=True) indexed with numpy at the same cells, byte for byte."""
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


def _tensor(a, dtype, device):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a).astype(dtype)).to(device)


def _check(dimg, master, host, rows, cols, k, as_float, what, dtype=np.int64):
    got = dimg.read_values(master, _tensor(rows, dtype, dimg.device), _tensor(cols, dtype, dimg.device), element=k, as_float=as_float)
    want = host[rows, cols]
    assert got.is_cuda and tuple(got.shape) == want.shape and str(got.dtype).endswith(host.dtype.name), what
    assert np.array_equal(_bytes(got), _bytes(want)), what
    return got


def _corner_and_tile_points(spec, rng, n_random):
    """The four corners, every tile's first and last cell inside the raster, and n_random seeded random cells."""
    R, Cc = spec.tile_rows, spec.tile_cols
    rows = [0, 0, spec.n_rows - 1, spec.n_rows - 1]
    cols = [0, spec.n_cols - 1, 0, spec.n_cols - 1]
    for tr in range(spec.tiles_down):
        for tc in range(spec.tiles_across):
            rows += [tr * R, min((tr + 1) * R, spec.n_rows) - 1]
            cols += [tc * Cc, min((tc + 1) * Cc, spec.n_cols) - 1]
    rows = np.concatenate([np.array(rows), rng.integers(0, spec.n_rows, n_random)])
    cols = np.concatenate([np.array(cols), rng.integers(0, spec.n_cols, n_random)])
    return rows, cols


@pytest.mark.gpu
def test_reference_files_read_as_the_host_reads_them(g4):
    from gridfour_b200 import gvrs

    n_files = 0
    for name, image in sample_files().items():
        img = gvrs.GvrsImage.parse(image)
        s = img.spec
        master = _master(g4, s.codecs)
        dimg = img.to_device()
        rows, cols = _corner_and_tile_points(s, np.random.default_rng(n_files), 2000)
        for k, e in enumerate(s.elements):
            for as_float in _float_modes(e):
                host = img.read_raster(master, element=k, crop=True, as_float=as_float)
                _check(dimg, master, host, rows, cols, k, as_float, (name, k, as_float))
        n_files += 1
    assert n_files == 17


# ---- written images -----------------------------------------------------------------------------------------------------
TR, TC = 20, 22          # tile size: the tile columns are not a multiple of 4, so tile edges fall at every residue
ROWS, COLS = 95, 127     # 5 x 6 tiles, the last row and column of tiles partial
DROP = (1, 8, 29)        # tiles left out of the directory (29 is the partial corner tile)


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
            s[30:45, 40:70] = -9999
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


def _write(g4, master, spec, grids, drop=DROP):
    from gridfour_b200 import gvrs

    ctx = master._context()
    w = gvrs.GvrsWriter(spec, uuid=bytes(range(16)), time_modified=1700000000000)
    for name, rid, typ, content, desc in gvrs.codec_metadata(spec.codecs):
        w.add_metadata(name, rid, typ, content, desc)
    batches = [w._encode_element(master, e, g) for e, g in zip(spec.elements, grids)]
    drop = set(drop)
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
    for checksum in (True, False):
        for key, (kinds, codecs) in CASES.items():
            master = _master(g4, codecs)
            spec = gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(kinds), codecs, checksum=checksum)
            out[key, checksum] = (master, _write(g4, master, spec, _grids(oracle, kinds)))
    return out


def _point_sets():
    rng = np.random.default_rng(7)
    sets = {"one": (np.array([37]), np.array([50]))}
    u = rng.integers(0, ROWS, 40), rng.integers(0, COLS, 40)
    pick = rng.integers(0, 40, 300)
    sets["duplicates, unsorted"] = (u[0][pick], u[1][pick])
    sets["one tile"] = (rng.integers(2 * TR, 3 * TR, 100), rng.integers(3 * TC, 4 * TC, 100))
    rows, cols = [], []
    for t in range(5 * 6):
        tr, tc = divmod(t, 6)
        rows += [tr * TR, min((tr + 1) * TR, ROWS) - 1, tr * TR + 7]
        cols += [tc * TC, min((tc + 1) * TC, COLS) - 1, min(tc * TC + 13, COLS - 1)]
    perm = rng.permutation(len(rows))
    sets["every tile"] = (np.array(rows)[perm], np.array(cols)[perm])
    sets["last row and column"] = (np.concatenate([np.full(COLS, ROWS - 1), np.arange(ROWS)]),
                                   np.concatenate([np.arange(COLS), np.full(ROWS, COLS - 1)]))
    sets["random"] = (rng.integers(0, ROWS, 2000), rng.integers(0, COLS, 2000))
    return sets


def _touched(rows, cols):
    return np.unique((np.asarray(rows) // TR) * 6 + np.asarray(cols) // TC)


@pytest.mark.gpu
@pytest.mark.parametrize("checksum", [True, False])
@pytest.mark.parametrize("case", list(CASES))
def test_point_sets_equal_the_host_raster(g4, written, case, checksum):
    import torch

    master, img = written[case, checksum]
    dimg = img.to_device()
    assert int((dimg.status == G4_DECLINED).sum()) == len(DROP)
    for k, e in enumerate(img.spec.elements):
        for as_float in _float_modes(e):
            host = img.read_raster(master, element=k, crop=True, as_float=as_float)
            for name, (rows, cols) in _point_sets().items():
                what = (case, checksum, k, as_float, name)
                for dtype in (np.int64, np.int32):
                    _check(dimg, master, host, rows, cols, k, as_float, what + (dtype,), dtype)
                tiles = _touched(rows, cols)
                assert np.array_equal(dimg.lastTiles.cpu().numpy(), tiles), what
                assert dimg.lastStatus.cpu().tolist() == [G4_DECLINED if t in DROP else G4_OK for t in tiles], what
            rows, cols = _point_sets()["random"]
            want = host[rows, cols]
            # non-contiguous index tensors: every other entry of a longer tensor
            r2 = _tensor(np.repeat(rows, 2), np.int64, dimg.device)[::2]
            c2 = _tensor(np.repeat(cols, 2), np.int32, dimg.device)[1::2]
            assert not r2.is_contiguous() and not c2.is_contiguous()
            assert np.array_equal(_bytes(dimg.read_values(master, r2, c2, element=k, as_float=as_float)), _bytes(want))
            # multi-dimensional shapes keep their shape
            for shape in [(40, 50), (2, 10, 100), (2000, 1)]:
                got = dimg.read_values(master, _tensor(rows, np.int64, dimg.device).reshape(shape),
                                       _tensor(cols, np.int32, dimg.device).reshape(shape), element=k, as_float=as_float)
                assert tuple(got.shape) == shape and np.array_equal(_bytes(got), _bytes(want.reshape(shape))), (case, k, shape)
            # into a given tensor
            out = torch.empty(want.shape, dtype=got.dtype, device=dimg.device)
            assert dimg.read_values(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device), element=k,
                                    as_float=as_float, out=out) is out
            assert np.array_equal(_bytes(out), _bytes(want))
            # no points
            empty = torch.empty(0, dtype=torch.int64, device=dimg.device)
            got = dimg.read_values(master, empty, empty, element=k, as_float=as_float)
            assert got.shape == (0,) and got.dtype == out.dtype
            assert dimg.lastTiles.numel() == 0 and dimg.lastStatus.numel() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_points_agree_with_single_cell_blocks(g4, written, case):
    master, img = written[case, True]
    dimg = img.to_device()
    rng = np.random.default_rng(11)
    rows, cols = rng.integers(0, ROWS, 200), rng.integers(0, COLS, 200)
    for k, e in enumerate(img.spec.elements):
        for as_float in _float_modes(e):
            got = dimg.read_values(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device), element=k,
                                   as_float=as_float).cpu()
            for i, (r, c) in enumerate(zip(rows, cols)):
                block = dimg.read_block(master, int(r), int(c), 1, 1, element=k, as_float=as_float).cpu()
                assert np.array_equal(_bytes(got[i:i + 1]), _bytes(block.reshape(1))), (case, k, as_float, r, c)


@pytest.mark.gpu
def test_async_point_reads(g4, written):
    master, img = written["three", True]
    dimg = img.to_device()
    ctx = dimg.context
    host = img.read_raster(master, element=2, crop=True, as_float=True)
    sets = _point_sets()
    ctx.set_async(True)
    try:
        outs = [(rows, cols, dimg.read_values(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device),
                                              element=2, as_float=True)) for rows, cols in sets.values()]
        status = dimg.lastStatus
        ctx.synchronize()
    finally:
        ctx.set_async(False)
    for rows, cols, got in outs:
        assert np.array_equal(_bytes(got), _bytes(host[rows, cols]))
    assert status.cpu().tolist() == [G4_DECLINED if t in DROP else G4_OK for t in _touched(*sets["random"])]


@pytest.mark.gpu
def test_many_tiles(g4, oracle):
    import torch

    from gridfour_b200 import gvrs

    rows_, cols_, tr, tc = 600, 600, 2, 2    # 90,000 tiles: more than 65,536, so the compaction takes several rounds
    codecs = ["GvrsHuffman", "GvrsDeflate"]
    master = _master(g4, codecs)
    spec = gvrs.GvrsSpec(rows_, cols_, tr, tc, _elements(["int"]), codecs, checksum=False)
    drop = range(1000, 90000, 997)
    img = _write(g4, master, spec, _grids(oracle, ["int"], rows_, cols_), drop=drop)
    host = img.read_raster(master, crop=True)
    dimg = img.to_device()
    rng = np.random.default_rng(5)
    n = 1 << 20
    rows, cols = rng.integers(0, rows_, n), rng.integers(0, cols_, n)
    got = dimg.read_values(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int32, dimg.device))
    assert np.array_equal(got.cpu().numpy(), host[rows, cols])
    tiles = np.unique((rows // tr) * (cols_ // tc) + cols // tc)
    assert dimg.lastTiles.numel() == len(tiles) > 65536
    assert np.array_equal(dimg.lastTiles.cpu().numpy(), tiles)
    dropped = set(drop)
    assert dimg.lastStatus.cpu().tolist() == [G4_DECLINED if t in dropped else G4_OK for t in tiles]
    # a second call on the same context: the compaction left the flags clear
    few = torch.tensor([[0, 0], [599, 599], [301, 2]], dtype=torch.int64, device=dimg.device)
    got = dimg.read_values(master, few[:, 0], few[:, 1])
    assert got.cpu().tolist() == [int(host[r, c]) for r, c in few.cpu().tolist()]
    assert dimg.lastTiles.cpu().tolist() == [0, 150 * 300 + 1, 299 * 300 + 299]


def _payload_location(img, t, element=0):
    """File offset and length of element `element` of tile t, read off the record on the host."""
    pos = img.tile_directory()[t] + 4
    for _ in range(element):
        pos += 4 + struct.unpack_from("<i", img.image, pos)[0]
    return pos + 4, struct.unpack_from("<i", img.image, pos)[0]


@pytest.mark.gpu
def test_a_malformed_payload_fails_only_its_tile(g4, oracle):
    from gridfour_b200 import gvrs

    codecs = ["GvrsHuffman", "GvrsDeflate", "LSOP12"]
    master = _master(g4, codecs)
    spec = gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(["int"]), codecs, checksum=False)
    img = _write(g4, master, spec, _grids(oracle, ["int"]), drop=())
    clean = img.read_raster(master, crop=True)
    victim = 2 * spec.tiles_across + 3   # tile row 2, tile column 3
    off, ln = _payload_location(img, victim)
    assert ln < 4 * TR * TC              # a codec packing, not a raw tile
    bad = bytearray(img.image)
    bad[off] = 200                       # packing[0]: no codec has that index (CodecMaster.decode throws)
    dimg = gvrs.GvrsImage.parse(bytes(bad)).to_device()
    for name, (rows, cols) in _point_sets().items():
        tiles = _touched(rows, cols)
        r, c = _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device)
        if victim in tiles:
            with pytest.raises(g4.FormatError):
                dimg.read_values(master, r, c)
            st = dimg.lastStatus.cpu().numpy()
            assert st[list(tiles).index(victim)] == G4_ERR_FORMAT and np.count_nonzero(st) == 1, name
        else:
            assert np.array_equal(dimg.read_values(master, r, c).cpu().numpy(), clean[rows, cols]), name


@pytest.mark.gpu
def test_a_value_checksum_mismatch_warns_and_delivers(g4, oracle):
    from gridfour_b200 import gvrs

    master = _master(g4, ["LSOP12"])
    master.getEncoder("LSOP12").setValueChecksumEnabled(True)
    rows_, cols_, tr, tc = 180, 240, 60, 80
    grid = oracle.terrain_i32(900, 1200, rows_, cols_)
    spec = gvrs.GvrsSpec(rows_, cols_, tr, tc, [gvrs.ElementSpec.integer("z")], ["LSOP12"], checksum=False)
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
    rng = np.random.default_rng(3)
    rows, cols = rng.integers(0, rows_, 500), rng.integers(0, cols_, 500)
    with pytest.warns(g4.ValueChecksumWarning):
        got = dimg.read_values(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device))
    assert np.array_equal(got.cpu().numpy(), grid[rows, cols])
    tiles = dimg.lastTiles.cpu().tolist()
    assert tiles == list(range(9))
    assert dimg.lastStatus.cpu().tolist() == [G4_CHECKSUM_MISMATCH if t == victim else G4_OK for t in tiles]
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        other = (victim + 1) % 9
        r, c = divmod(other, 3)
        rr, cc = r * tr + rng.integers(0, tr, 50), c * tc + rng.integers(0, tc, 50)
        got = dimg.read_values(master, _tensor(rr, np.int64, dimg.device), _tensor(cc, np.int64, dimg.device))
        assert np.array_equal(got.cpu().numpy(), grid[rr, cc])


@pytest.mark.gpu
def test_points_outside_the_raster_are_refused(g4, written):
    import torch

    from gridfour_b200 import _lib

    master, img = written["icf", True]
    dimg = img.to_device()
    dev = dimg.device
    L, ctx, spec = _lib.lib(), dimg.context, img.spec
    icf = spec.elements[0].icf.desc()
    bad_icf = _lib.IcfDesc()
    bad_icf.scale = 0.0
    good = (np.array([0, 25, ROWS - 1]), np.array([0, 30, COLS - 1]))   # tiles 0, 7 and 29 (absent)
    outside = {"negative row": (np.array([3, -1]), np.array([3, 3])), "negative column": (np.array([3, 3]), np.array([3, -2])),
               "row == n_rows": (np.array([ROWS]), np.array([0])), "column == n_cols": (np.array([0]), np.array([COLS])),
               "fill margin": (np.array([ROWS + 2]), np.array([COLS + 3]))}   # inside the last tiles, outside the raster
    assert ROWS + 2 < spec.tiles_down * TR and COLS + 3 < spec.tiles_across * TC
    for name, (rows, cols) in outside.items():
        with pytest.raises(ValueError):
            dimg.read_values(master, _tensor(rows, np.int64, dev), _tensor(cols, np.int64, dev))
    with pytest.raises(ValueError):   # indices in host memory
        dimg.read_values(master, torch.from_numpy(good[0]), _tensor(good[1], np.int64, dev))
    with pytest.raises(ValueError):
        dimg.read_values(master, _tensor(good[0], np.int64, dev), torch.from_numpy(good[1]))
    if torch.cuda.device_count() > 1:
        other = torch.device("cuda", (dev.index + 1) % torch.cuda.device_count())
        with pytest.raises(ValueError):
            dimg.read_values(master, _tensor(good[0], np.int64, other), _tensor(good[1], np.int64, other))
    with pytest.raises(ValueError):   # float indices
        dimg.read_values(master, _tensor(good[0], np.float32, dev), _tensor(good[1], np.int64, dev))
    with pytest.raises(ValueError):   # shapes differ
        dimg.read_values(master, _tensor(good[0], np.int64, dev), _tensor(good[1][:2], np.int64, dev))
    with pytest.raises(ValueError):   # out of the wrong dtype
        dimg.read_values(master, _tensor(good[0], np.int64, dev), _tensor(good[1], np.int64, dev), as_float=True,
                         out=torch.empty(3, dtype=torch.int32, device=dev))
    with pytest.raises(ValueError):
        dimg.read_values(master, _tensor(good[0], np.int64, dev), _tensor(good[1], np.int64, dev), element=1)

    # the C call: G4_ERR_ARG, and the sentinel in `out` is left as it was
    n_tiles = spec.tiles_down * spec.tiles_across
    tiles = torch.empty(n_tiles, dtype=torch.int32, device=dev)
    st = torch.empty(n_tiles, dtype=torch.int32, device=dev)

    def band(elem=G4_ELEM_ICF, down=spec.tiles_down):
        b = _lib.BandDesc()
        b.elem_type, b.tile_rows, b.tile_cols, b.tiles_down, b.tiles_across = elem, TR, TC, down, spec.tiles_across
        b.grid_pitch = spec.tiles_across * TC
        return b

    def call(rows, cols, b=None, d=icf, n_rows=ROWS, n_cols=COLS, n=None, rows_ptr=None):
        r = rows if isinstance(rows, torch.Tensor) else _tensor(rows, np.int64, dev)
        c = _tensor(cols, np.int64, dev)
        out = torch.full((len(cols),), -12345.0, dtype=torch.float32, device=dev)
        k = C.c_int32(-1)
        rc = L.g4_decode_points(ctx._h, C.byref(master._native_list()), C.byref(b or band()), None if d is None else C.byref(d),
                                dimg.image.data_ptr(), int(dimg.image.numel()), dimg.payload_off[0].data_ptr(), dimg.lens[0].data_ptr(),
                                dimg.status.data_ptr(), 0, n_rows, n_cols, len(cols) if n is None else n,
                                r.data_ptr() if rows_ptr is None else rows_ptr, c.data_ptr(), out.data_ptr(), tiles.data_ptr(),
                                st.data_ptr(), C.byref(k))
        return rc, out, k.value

    rc, out, k = call(*good)
    want = img.read_raster(master, crop=True, as_float=True)[good]
    want[2] = 0.0   # tile 29 is absent: it reads as the fill_bits passed (0)
    assert rc == G4_OK and k == 3 and np.array_equal(_bytes(out), _bytes(want))
    rc, out, k = call(*good, b=band(G4_ELEM_I32), d=None)          # the codes
    assert rc == G4_OK and k == 3
    host_rows = torch.from_numpy(good[0].astype(np.int64))
    cases = [call(rows, cols) for rows, cols in outside.values()]
    cases += [call(host_rows, good[1]),                                       # indices in host memory
              call(*good, rows_ptr=0),                                        # a null pointer
              call(*good, n=-1),                                              # a negative count
              call(*good, d=bad_icf), call(*good, d=None),                    # an invalid descriptor, none for ICF
              call(*good, b=band(G4_ELEM_I32)),                               # a descriptor for a non-ICF element
              call(*good, b=band(7), d=None), call(*good, b=band(down=0)),    # bad raster
              call(*good, n_rows=spec.tiles_down * TR + 1), call(*good, n_cols=spec.tiles_across * TC + 1),  # extent > grid
              call(*good, n_rows=0)]
    for i, (rc, out, k) in enumerate(cases):
        assert rc == G4_ERR_ARG and k == 0, i
        assert (out == -12345.0).all(), i
    rc, out, k = call(*good)   # the context is unharmed
    assert rc == G4_OK and k == 3
    rc, out, k = call(np.array([], dtype=np.int64), np.array([], dtype=np.int64), rows_ptr=0)   # no points: nothing needed
    assert rc == G4_OK and k == 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["int", "float"])
def test_point_reads_add_three_launches_to_the_band_decode(g4, written, case):
    import torch

    from gridfour_b200 import _lib

    master, img = written[case, True]
    dimg = img.to_device()
    ctx = dimg.context
    rng = np.random.default_rng(2)
    rows, cols = rng.integers(2 * TR, 4 * TR, 300), rng.integers(0, COLS, 300)   # tile rows 2 and 3: every tile present
    r, c = _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device)
    n0 = ctx.launch_count
    got = dimg.read_values(master, r, c)
    n1 = ctx.launch_count
    idx = dimg.lastTiles.long()
    K = idx.numel()
    assert K == 12
    off = dimg.payload_off[0][idx].contiguous()
    lens = dimg.lens[0][idx].contiguous()
    band = _lib.BandDesc()
    band.elem_type = G4_ELEM_F32 if case == "float" else G4_ELEM_I32
    band.tile_rows, band.tile_cols, band.tiles_down, band.tiles_across, band.grid_pitch = TR, TC, K, 1, TC
    grid = torch.empty((K * TR, TC), dtype=torch.float32 if case == "float" else torch.int32, device=dimg.device)
    status = torch.empty(K, dtype=torch.int32, device=dimg.device)
    assert _lib.lib().g4_decode_tiles_bounded(ctx._h, C.byref(master._native_list()), C.byref(band), G4_MEM_DEVICE, dimg.image.data_ptr(),
                                              int(dimg.image.numel()), off.data_ptr(), lens.data_ptr(), grid.data_ptr(),
                                              status.data_ptr()) == G4_OK
    n2 = ctx.launch_count
    assert (n1 - n0) - (n2 - n1) == 3
    slot = {t: k for k, t in enumerate(dimg.lastTiles.cpu().tolist())}
    g = grid.cpu().numpy().reshape(K, TR, TC)
    want = np.array([g[slot[(a // TR) * 6 + b // TC], a % TR, b % TC] for a, b in zip(rows, cols)])
    assert np.array_equal(_bytes(got), _bytes(want))
    empty = torch.empty(0, dtype=torch.int64, device=dimg.device)
    n3 = ctx.launch_count
    dimg.read_values(master, empty, empty)
    assert ctx.launch_count == n3
