"""Block reads from a GVRS file image resident on the GPU (GvrsDeviceImage.read_blocks, g4_decode_blocks): every block equals
the host read_raster(crop=True) sliced with numpy at the same window, byte for byte."""
import ctypes as C
import struct

import numpy as np
import pytest

from gvrs_common import sample_files

G4_OK, G4_DECLINED = 0, 1
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


def _want(host, rows, cols, h, w):
    return np.stack([host[r:r + h, c:c + w] for r, c in zip(rows, cols)]) if len(rows) else np.empty((0, h, w), host.dtype)


def _covered(rows, cols, h, w, tr, tc, tiles_across):
    t = set()
    for r, c in zip(rows, cols):
        for a in range(r // tr, (r + h - 1) // tr + 1):
            for b in range(c // tc, (c + w - 1) // tc + 1):
                t.add(a * tiles_across + b)
    return np.array(sorted(t), dtype=np.int64)


def _check(dimg, master, host, rows, cols, h, w, k, as_float, what, dtype=np.int64):
    got = dimg.read_blocks(master, _tensor(rows, dtype, dimg.device), _tensor(cols, dtype, dimg.device), h, w, element=k,
                           as_float=as_float)
    want = _want(host, rows, cols, h, w)
    assert got.is_cuda and tuple(got.shape) == want.shape and str(got.dtype).endswith(host.dtype.name), what
    assert np.array_equal(_bytes(got), _bytes(want)), what
    spec = dimg.spec
    tiles = _covered(rows, cols, h, w, spec.tile_rows, spec.tile_cols, spec.tiles_across)
    assert np.array_equal(dimg.lastTiles.cpu().numpy(), tiles), what
    return got


def _random_blocks(rng, n, h, w, n_rows, n_cols):
    return rng.integers(0, n_rows - h + 1, n), rng.integers(0, n_cols - w + 1, n)


@pytest.mark.gpu
def test_reference_files_read_as_the_host_reads_them(g4):
    from gridfour_b200 import gvrs

    n_files = 0
    for name, image in sample_files().items():
        img = gvrs.GvrsImage.parse(image)
        s = img.spec
        master = _master(g4, s.codecs)
        dimg = img.to_device()
        rng = np.random.default_rng(n_files)
        shapes = [(1, 1), (3, 5), (min(s.tile_rows, s.n_rows), min(s.tile_cols, s.n_cols)),
                  (min(2 * s.tile_rows + 3, s.n_rows), min(2 * s.tile_cols + 5, s.n_cols)), (s.n_rows, s.n_cols)]
        for k, e in enumerate(s.elements):
            for as_float in _float_modes(e):
                host = img.read_raster(master, element=k, crop=True, as_float=as_float)
                for h, w in shapes:
                    rows, cols = _random_blocks(rng, 40 if h * w < 10 ** 6 else 1, h, w, s.n_rows, s.n_cols)
                    _check(dimg, master, host, rows, cols, h, w, k, as_float, (name, k, as_float, h, w))
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
            v = oracle.terrain_f32(200 + k, 50, rows, cols)
            v[10:25, 70:90] = np.nan
            out.append(v)
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
            "float": lambda k: gvrs.ElementSpec.floating("e%d" % k, fill_value=float("nan")),
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
    for key, (kinds, codecs) in CASES.items():
        master = _master(g4, codecs)
        spec = gvrs.GvrsSpec(ROWS, COLS, TR, TC, _elements(kinds), codecs, checksum=True)
        out[key] = (master, _write(g4, master, spec, _grids(oracle, kinds)))
    return out


def _block_sets():
    """(n_rows, n_cols, rows, cols) per name: every width residue mod 4, tile-sized blocks at tile origins, blocks over
    3 x 3 tiles and more, overlapping, duplicate and unordered blocks, and the whole raster."""
    rng = np.random.default_rng(7)
    sets = {}
    for h, w in [(1, 1), (1, 2), (2, 3), (5, 7), (4, 4), (3, 8), (9, 13), (6, 16), (17, 21)]:
        sets["%dx%d" % (h, w)] = (h, w) + _random_blocks(rng, 60, h, w, ROWS, COLS)
    origins = [(tr * TR, tc * TC) for tr in range(ROWS // TR) for tc in range(COLS // TC)]   # whole tiles inside the raster
    perm = rng.permutation(len(origins))
    sets["tile at tile origins"] = (TR, TC, np.array([origins[i][0] for i in perm]), np.array([origins[i][1] for i in perm]))
    sets["3 x 3 tiles and more"] = (3 * TR - 1, 3 * TC + 5) + _random_blocks(rng, 12, 3 * TR - 1, 3 * TC + 5, ROWS, COLS)
    r, c = _random_blocks(rng, 10, 11, 30, ROWS, COLS)
    pick = rng.integers(0, 10, 50)
    sets["overlapping, duplicate, unordered"] = (11, 30, r[pick], c[pick])
    sets["whole raster"] = (ROWS, COLS, np.array([0]), np.array([0]))
    sets["last row and column"] = (2, 5, np.array([ROWS - 2, 0, ROWS - 2, 40]), np.array([COLS - 5, COLS - 5, 0, COLS - 5]))
    return sets


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_block_sets_equal_the_host_raster(g4, written, case):
    import torch

    master, img = written[case]
    dimg = img.to_device()
    assert int((dimg.status == G4_DECLINED).sum()) == len(DROP)
    for k, e in enumerate(img.spec.elements):
        for as_float in _float_modes(e):
            host = img.read_raster(master, element=k, crop=True, as_float=as_float)
            for name, (h, w, rows, cols) in _block_sets().items():
                what = (case, k, as_float, name)
                for dtype in (np.int64, np.int32):
                    _check(dimg, master, host, rows, cols, h, w, k, as_float, what + (dtype,), dtype)
                tiles = dimg.lastTiles.cpu().tolist()
                assert dimg.lastStatus.cpu().tolist() == [G4_DECLINED if t in DROP else G4_OK for t in tiles], what
            # 1 x 1 blocks are points
            h, w, rows, cols = _block_sets()["1x1"]
            r, c = _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device)
            got = dimg.read_blocks(master, r, c, 1, 1, element=k, as_float=as_float)
            assert np.array_equal(_bytes(got.reshape(-1)), _bytes(dimg.read_values(master, r, c, element=k, as_float=as_float)))
            # into a given tensor
            h, w, rows, cols = _block_sets()["9x13"]
            out = torch.empty((len(rows), h, w), dtype=got.dtype, device=dimg.device)
            assert dimg.read_blocks(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device), h, w,
                                    element=k, as_float=as_float, out=out) is out
            assert np.array_equal(_bytes(out), _bytes(_want(host, rows, cols, h, w)))
            # no blocks
            empty = torch.empty(0, dtype=torch.int64, device=dimg.device)
            got = dimg.read_blocks(master, empty, empty, 3, 4, element=k, as_float=as_float)
            assert tuple(got.shape) == (0, 3, 4) and got.dtype == out.dtype
            assert dimg.lastTiles.numel() == 0 and dimg.lastStatus.numel() == 0


@pytest.mark.gpu
def test_blocks_agree_with_read_block(g4, written):
    master, img = written["three"]
    dimg = img.to_device()
    rng = np.random.default_rng(11)
    for k, e in enumerate(img.spec.elements):
        for as_float in _float_modes(e):
            for h, w in [(1, 1), (7, 5), (TR, TC), (30, 50)]:
                rows, cols = _random_blocks(rng, 20, h, w, ROWS, COLS)
                got = dimg.read_blocks(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device), h, w,
                                       element=k, as_float=as_float).cpu()
                for i, (r, c) in enumerate(zip(rows, cols)):
                    block = dimg.read_block(master, int(r), int(c), h, w, element=k, as_float=as_float).cpu()
                    assert np.array_equal(_bytes(got[i]), _bytes(block)), (k, as_float, h, w, r, c)


@pytest.mark.gpu
def test_async_block_reads(g4, written):
    master, img = written["three"]
    dimg = img.to_device()
    ctx = dimg.context
    host = img.read_raster(master, element=2, crop=True, as_float=True)
    sets = _block_sets()
    ctx.set_async(True)
    try:
        outs = [(h, w, rows, cols, dimg.read_blocks(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device),
                                                    h, w, element=2, as_float=True)) for h, w, rows, cols in sets.values()]
        status = dimg.lastStatus
        ctx.synchronize()
    finally:
        ctx.set_async(False)
    for h, w, rows, cols, got in outs:
        assert np.array_equal(_bytes(got), _bytes(_want(host, rows, cols, h, w)))
    h, w, rows, cols = list(sets.values())[-1]
    assert status.cpu().tolist() == [G4_DECLINED if t in DROP else G4_OK for t in _covered(rows, cols, h, w, TR, TC, 6)]


@pytest.mark.gpu
def test_many_tiles(g4, oracle):
    import torch

    from gridfour_b200 import gvrs

    rows_, cols_, tr, tc = 600, 600, 2, 2    # 90,000 tiles: the compaction takes several rounds; a quad spans up to 3 tiles
    codecs = ["GvrsHuffman", "GvrsDeflate"]
    master = _master(g4, codecs)
    spec = gvrs.GvrsSpec(rows_, cols_, tr, tc, _elements(["int"]), codecs, checksum=False)
    drop = range(1000, 90000, 997)
    img = _write(g4, master, spec, _grids(oracle, ["int"], rows_, cols_), drop=drop)
    host = img.read_raster(master, crop=True)
    dimg = img.to_device()
    rng = np.random.default_rng(5)
    dropped = set(drop)
    for h, w, n in [(9, 7, 4096), (1, 5, 20000), (3, 3, 30000), (rows_, cols_, 1)]:
        rows, cols = _random_blocks(rng, n, h, w, rows_, cols_)
        got = dimg.read_blocks(master, _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int32, dimg.device), h, w)
        assert np.array_equal(got.cpu().numpy(), _want(host, rows, cols, h, w)), (h, w)
        tiles = _covered(rows, cols, h, w, tr, tc, cols_ // tc)
        assert dimg.lastTiles.numel() == len(tiles) > 16384, (h, w)
        assert np.array_equal(dimg.lastTiles.cpu().numpy(), tiles), (h, w)
        assert dimg.lastStatus.cpu().tolist() == [G4_DECLINED if t in dropped else G4_OK for t in tiles], (h, w)
    # a second call on the same context: the compaction left the flags clear
    few = torch.tensor([[0, 0], [595, 596], [301, 2]], dtype=torch.int64, device=dimg.device)
    got = dimg.read_blocks(master, few[:, 0], few[:, 1], 4, 3)
    assert np.array_equal(got.cpu().numpy(), _want(host, [0, 595, 301], [0, 596, 2], 4, 3))
    assert np.array_equal(dimg.lastTiles.cpu().numpy(), _covered([0, 595, 301], [0, 596, 2], 4, 3, tr, tc, cols_ // tc))
    assert dimg.lastTiles.numel() == 4 + 6 + 6


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
    n_hit = 0
    for name, (h, w, rows, cols) in _block_sets().items():
        tiles = list(_covered(rows, cols, h, w, TR, TC, 6))
        r, c = _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device)
        if victim in tiles:
            n_hit += 1
            with pytest.raises(g4.FormatError):
                dimg.read_blocks(master, r, c, h, w)
            st = dimg.lastStatus.cpu().numpy()
            assert st[tiles.index(victim)] == G4_ERR_FORMAT and np.count_nonzero(st) == 1, name
        else:
            assert np.array_equal(dimg.read_blocks(master, r, c, h, w).cpu().numpy(), _want(clean, rows, cols, h, w)), name
    assert n_hit >= 3


@pytest.mark.gpu
def test_blocks_outside_the_raster_are_refused(g4, written):
    import torch

    from gridfour_b200 import _lib

    master, img = written["icf"]
    dimg = img.to_device()
    dev = dimg.device
    L, ctx, spec = _lib.lib(), dimg.context, img.spec
    icf = spec.elements[0].icf.desc()
    bad_icf = _lib.IcfDesc()
    bad_icf.scale = 0.0
    H, W = 5, 6
    good = (np.array([0, 25, ROWS - H]), np.array([0, 30, COLS - W]))   # tiles 0, 7 and 29 (absent)
    outside = {"negative row": (np.array([3, -1]), np.array([3, 3])), "negative column": (np.array([3, 3]), np.array([3, -2])),
               "one row past": (np.array([ROWS - H + 1]), np.array([0])), "one column past": (np.array([0]), np.array([COLS - W + 1])),
               "fill margin": (np.array([ROWS - 2]), np.array([COLS - 3]))}   # inside the last tiles, outside the raster
    assert ROWS + 3 < spec.tiles_down * TR and COLS + 3 < spec.tiles_across * TC
    for name, (rows, cols) in outside.items():
        with pytest.raises(ValueError):
            dimg.read_blocks(master, _tensor(rows, np.int64, dev), _tensor(cols, np.int64, dev), H, W)
    with pytest.raises(ValueError):   # indices in host memory
        dimg.read_blocks(master, torch.from_numpy(good[0]), _tensor(good[1], np.int64, dev), H, W)
    with pytest.raises(ValueError):
        dimg.read_blocks(master, _tensor(good[0], np.int64, dev), torch.from_numpy(good[1]), H, W)
    with pytest.raises(ValueError):   # float indices
        dimg.read_blocks(master, _tensor(good[0], np.float32, dev), _tensor(good[1], np.int64, dev), H, W)
    with pytest.raises(ValueError):   # lengths differ
        dimg.read_blocks(master, _tensor(good[0], np.int64, dev), _tensor(good[1][:2], np.int64, dev), H, W)
    with pytest.raises(ValueError):   # 2-D indices
        dimg.read_blocks(master, _tensor(good[0], np.int64, dev).reshape(3, 1), _tensor(good[1], np.int64, dev).reshape(3, 1), H, W)
    for h, w in [(0, W), (H, 0), (-1, W)]:
        with pytest.raises(ValueError):
            dimg.read_blocks(master, _tensor(good[0], np.int64, dev), _tensor(good[1], np.int64, dev), h, w)
    with pytest.raises(ValueError):   # out of the wrong dtype, shape or layout
        dimg.read_blocks(master, _tensor(good[0], np.int64, dev), _tensor(good[1], np.int64, dev), H, W, as_float=True,
                         out=torch.empty((3, H, W), dtype=torch.int32, device=dev))
    with pytest.raises(ValueError):
        dimg.read_blocks(master, _tensor(good[0], np.int64, dev), _tensor(good[1], np.int64, dev), H, W, as_float=True,
                         out=torch.empty((3, H, W + 1), dtype=torch.float32, device=dev))
    with pytest.raises(ValueError):
        dimg.read_blocks(master, _tensor(good[0], np.int64, dev), _tensor(good[1], np.int64, dev), H, W, as_float=True,
                         out=torch.empty((3, W, H), dtype=torch.float32, device=dev).transpose(1, 2))
    with pytest.raises(ValueError):
        dimg.read_blocks(master, _tensor(good[0], np.int64, dev), _tensor(good[1], np.int64, dev), H, W, element=1)

    # the C call: G4_ERR_ARG with K = 0, and the sentinel in `out` is left as it was
    n_tiles = spec.tiles_down * spec.tiles_across
    tiles = torch.empty(n_tiles, dtype=torch.int32, device=dev)
    st = torch.empty(n_tiles, dtype=torch.int32, device=dev)

    def band(elem=G4_ELEM_ICF, down=spec.tiles_down):
        b = _lib.BandDesc()
        b.elem_type, b.tile_rows, b.tile_cols, b.tiles_down, b.tiles_across = elem, TR, TC, down, spec.tiles_across
        b.grid_pitch = spec.tiles_across * TC
        return b

    def call(rows, cols, b=None, d=icf, n_rows=ROWS, n_cols=COLS, n=None, h=H, w=W, rows_ptr=None, out_ptr=None, tiles_ptr=None):
        r = rows if isinstance(rows, torch.Tensor) else _tensor(rows, np.int64, dev)
        c = _tensor(cols, np.int64, dev)
        out = torch.full((max(len(cols), 1) * H * W,), -12345.0, dtype=torch.float32, device=dev)
        host_out = torch.full_like(out, -12345.0, device="cpu")
        k = C.c_int32(-1)
        ptr = {None: out.data_ptr(), "host": host_out.data_ptr()}.get(out_ptr, out_ptr)
        rc = L.g4_decode_blocks(ctx._h, C.byref(master._native_list()), C.byref(b or band()), None if d is None else C.byref(d),
                                dimg.image.data_ptr(), int(dimg.image.numel()), dimg.payload_off[0].data_ptr(), dimg.lens[0].data_ptr(),
                                dimg.status.data_ptr(), 0, n_rows, n_cols, len(cols) if n is None else n,
                                r.data_ptr() if rows_ptr is None else rows_ptr, c.data_ptr(), h, w, ptr,
                                tiles.data_ptr() if tiles_ptr is None else tiles_ptr, st.data_ptr(), C.byref(k))
        torch.cuda.synchronize(dev)
        return rc, out, k.value, host_out

    host = img.read_raster(master, crop=True, as_float=True)
    rc, out, k, _ = call(*good)
    want = _want(host, good[0], good[1], H, W)
    want[2] = 0.0   # tile 29 is absent: it reads as the fill_bits passed (0)
    assert rc == G4_OK and k == 3 and np.array_equal(_bytes(out), _bytes(want).reshape(-1))
    assert tiles[:3].cpu().tolist() == [0, 7, 29] and st[:3].cpu().tolist() == [G4_OK, G4_OK, G4_DECLINED]
    rc, out, k, _ = call(*good, b=band(G4_ELEM_I32), d=None)          # the codes
    assert rc == G4_OK and k == 3
    host_rows = torch.from_numpy(good[0].astype(np.int64))
    cases = [call(rows, cols) for rows, cols in outside.values()]
    cases += [call(host_rows, good[1]),                                       # indices in host memory
              call(*good, rows_ptr=0),                                        # null pointers
              call(*good, out_ptr=0), call(*good, tiles_ptr=0),
              call(*good, h=0), call(*good, w=0),                             # empty blocks
              call(*good, n=-1),                                              # a negative count
              call(*good, h=1 << 32, w=1 << 31),                              # n * h * w overflows int64
              call(*good, d=bad_icf), call(*good, d=None),                    # an invalid descriptor, none for ICF
              call(*good, b=band(G4_ELEM_I32)),                               # a descriptor for a non-ICF element
              call(*good, b=band(7), d=None), call(*good, b=band(down=0)),    # bad raster
              call(*good, n_rows=spec.tiles_down * TR + 1), call(*good, n_cols=spec.tiles_across * TC + 1),  # extent > grid
              call(*good, n_rows=0),
              call(*good, h=ROWS + 1), call(*good, w=COLS + 1)]               # blocks larger than the raster
    for i, (rc, out, k, _) in enumerate(cases):
        assert rc == G4_ERR_ARG and k == 0, i
        assert (out == -12345.0).all(), i
    rc, _, k, host_out = call(*good, out_ptr="host")                         # `out` in host memory
    assert rc == G4_ERR_ARG and k == 0 and (host_out == -12345.0).all()
    rc, out, k, _ = call(*good)   # the context is unharmed
    assert rc == G4_OK and k == 3 and np.array_equal(_bytes(out), _bytes(want).reshape(-1))
    rc, out, k, _ = call(np.array([], dtype=np.int64), np.array([], dtype=np.int64), rows_ptr=0, out_ptr=0)   # no blocks
    assert rc == G4_OK and k == 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["int", "float"])
def test_block_reads_add_three_launches_to_the_band_decode(g4, written, case):
    import torch

    from gridfour_b200 import _lib

    master, img = written[case]
    dimg = img.to_device()
    ctx = dimg.context
    rng = np.random.default_rng(2)
    h, w = 13, 30
    rows, cols = rng.integers(2 * TR, 4 * TR - h + 1, 40), rng.integers(0, COLS - w + 1, 40)   # tile rows 2 and 3: every tile present
    r, c = _tensor(rows, np.int64, dimg.device), _tensor(cols, np.int64, dimg.device)
    n0 = ctx.launch_count
    got = dimg.read_blocks(master, r, c, h, w)
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
    mosaic = np.concatenate([np.concatenate([g[slot[a * 6 + b]] for b in range(6)], axis=1) for a in (2, 3)], axis=0)
    want = np.stack([mosaic[a - 2 * TR:a - 2 * TR + h, b:b + w] for a, b in zip(rows, cols)])
    assert np.array_equal(_bytes(got), _bytes(want))
    empty = torch.empty(0, dtype=torch.int64, device=dimg.device)
    n3 = ctx.launch_count
    dimg.read_blocks(master, empty, empty, h, w)
    assert ctx.launch_count == n3
