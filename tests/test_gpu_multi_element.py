"""Tile records of rasters with several elements per tile (RecordManager.writeTile / readTile, gvrs/RecordManager.java:386-516):
g4_pack_tile_records_multi / g4_unpack_tile_records_multi against a host restatement of the framing, the reference's
Sample08_MixedTypes file, and a three-element raster written and read end to end on the GPU.  Oracle: oracle/g4oracle
(CRC-32C, codecs)."""
import ctypes as C
import struct

import numpy as np
import pytest

from gvrs_common import sample_files, tile_record_parts

G4_OK, G4_DECLINED, G4_CHECKSUM_MISMATCH = 0, 1, 2
G4_ERR_ARG, G4_ERR_FORMAT, G4_ERR_CAPACITY, G4_ERR_UNSUPPORTED = -1, -2, -3, -5
ORACLE_IDS = {"GvrsHuffman": 0, "GvrsDeflate": 1, "GvrsFloat": 2, "GvrsCanonicalHuffman": 3, "LSOP12": 4}


@pytest.fixture(scope="module")
def g4():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import gridfour_b200

    return gridfour_b200


def test_records_bound_multi():
    from gridfour_b200 import _lib

    L = _lib.lib()
    assert L.g4_tile_records_bound_multi(10, 1, 1000) == L.g4_tile_records_bound(10, 1000) - 10 * 32 + 10 * 27
    assert L.g4_tile_records_bound_multi(3, 5, 77) == 77 + 3 * (23 + 20)
    assert L.g4_tile_records_bound_multi(3, 0, 77) == 0 and L.g4_tile_records_bound_multi(3, 65, 77) == 0
    assert L.g4_tile_records_bound_multi(-1, 2, 77) == 0


def host_record(tile_index, payloads, crc=None):
    """[size][2,0,0,0][tileIndex] then [len][bytes] per element, zero padding, [crc32c] -- the reference's framing."""
    from gridfour_b200 import gvrs

    content = struct.pack("<i", tile_index) + b"".join(struct.pack("<i", len(p)) + bytes(p) for p in payloads)
    rec = bytearray(gvrs.frame_record(gvrs.RECORD_TILE, content))
    if crc is not None:
        struct.pack_into("<I", rec, len(rec) - 4, crc(bytes(rec[:-4])))
    return bytes(rec)


def host_walk(image, content_pos, n_elements):
    """Element-major payload offsets and lengths of the [len][bytes] chain of every sound record (0 / 0 for absent tiles)."""
    n = len(content_pos)
    off = np.zeros((n_elements, n), np.uint64)
    lens = np.zeros((n_elements, n), np.uint32)
    for t, p in enumerate(content_pos):
        p = int(p)
        if not p:
            continue
        q = p + 4
        for e in range(n_elements):
            ln = struct.unpack_from("<i", image, q)[0]
            off[e, t], lens[e, t] = q + 4, ln
            q += 4 + ln
    return off, lens


def make_batch(rng, n_elements, n_tiles):
    """One arena per element: payload lengths 0..5000 with every residue mod 16, offsets at every residue mod 8."""
    arenas, offsets, lens, payloads = [], [], [], []
    for e in range(n_elements):
        ln = rng.integers(0, 5001, n_tiles)
        ln[:16] = np.arange(16) + 16 * rng.integers(0, 312, 16)
        ln[16:20] = [0, 1, 4, 5000]
        rng.shuffle(ln)
        arena, off, pl = bytearray(), [], []
        for t in range(n_tiles):
            arena += bytes((t + e - len(arena)) % 8 + 8 * int(rng.integers(0, 2)))  # offset residue (t + e) mod 8
            off.append(len(arena))
            p = rng.integers(0, 256, int(ln[t]), dtype=np.uint8).tobytes()
            pl.append(p)
            arena += p
        arena += bytes(5)
        arenas.append(np.frombuffer(bytes(arena), np.uint8))
        offsets.append(np.array(off, np.uint64))
        lens.append(ln.astype(np.uint32))
        payloads.append(pl)
    return arenas, offsets, lens, payloads


@pytest.mark.gpu
def test_sample08_mixed_types_byte_for_byte(g4, oracle):
    """The reference's two-element sample (one short, one float element): tile records framed by g4_pack_tile_records_multi,
    everything else written as tests/gvrs_common.rebuild writes it; the image is the reference file."""
    from gridfour_b200 import gvrs

    image = sample_files()["Sample08_MixedTypes.gvrs"]
    img = gvrs.GvrsImage.parse(image)
    assert len(img.spec.elements) == 2 and not img.spec.checksum
    ctx = g4.Context.default()
    w = gvrs.GvrsWriter(img.spec, uuid=img.uuid, time_modified=img.time_modified, version=img.version)
    order, tiles = [], []
    recs = img.records
    i = 0
    while i < len(recs):
        r = recs[i]
        if r.type_code == gvrs.RECORD_METADATA:
            rd = gvrs._Reader(r.body, 0)
            name = rd.utf()
            record_id, type_code, n = rd.take("<iB3xi")
            content = rd.raw(n)
            w.add_metadata(name, record_id, type_code, content, rd.utf(), size=r.size)
            i += 1
        elif r.type_code == gvrs.RECORD_TILE:
            j = i
            while j < len(recs) and recs[j].type_code == gvrs.RECORD_TILE:
                j += 1
            run = [tile_record_parts(t.body, 2) for t in recs[i:j]]
            assert [len(host_record(ti, parts)) for ti, parts in run] == [t.size for t in recs[i:j]]
            arenas, offsets, lens = [], [], []
            for e in range(2):
                arena, off = bytearray(), []
                for _, parts in run:
                    arena += bytes((-len(arena)) & 7)
                    off.append(len(arena))
                    arena += parts[e]
                arenas.append(bytes(arena) + bytes(8))
                offsets.append(off)
                lens.append([len(parts[e]) for _, parts in run])
            index = [ti for ti, _ in run]
            base = w.file_pos
            w.add_tile_records_multi(ctx, arenas, offsets, lens, tile_index=index)
            tiles.append((base, arenas, offsets, lens, index, run))
            i = j
        else:
            order.append("metadata" if r.type_code == gvrs.RECORD_METADATA_DIR else "tile")
            i += 1
    assert len(tiles) == 1 and len(tiles[0][5]) == 4
    assert w.finish(ctx, directory_order=tuple(order)) == image
    base, arenas, offsets, lens, index, run = tiles[0]
    got, pos = gvrs.pack_tile_records_multi(ctx, arenas, offsets, lens, base, True, tile_index=index)
    want = b"".join(host_record(ti, parts, oracle.crc32c) for ti, parts in run)
    assert got == want
    assert [int(p) for p in pos] == [r.content_pos for r in recs if r.type_code == gvrs.RECORD_TILE]


def _device_batches(g4, torch, arenas, offsets, lens):
    out = []
    for a, o, ln in zip(arenas, offsets, lens):
        t = torch.from_numpy(np.array(a)).cuda()
        out.append(g4.TileBatch(t, torch.from_numpy(o.astype(np.int64)).cuda(), torch.from_numpy(ln.astype(np.int32)).cuda(),
                                None, None, None, int(a.size), None))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n_elements", [1, 2, 3, 5, 8])
def test_framing_matches_host_restatement(g4, oracle, n_elements):
    import torch

    from gridfour_b200 import _lib, gvrs

    ctx = g4.Context.default()
    rng = np.random.default_rng(100 + n_elements)
    n = 300
    arenas, offsets, lens, payloads = make_batch(rng, n_elements, n)
    for base_pos, checksum, tile_index in ((0, True, None), (8, False, None), (4096, True, rng.permutation(n).astype(np.int32)),
                                           (1 << 33, True, None)):
        first = 7 if tile_index is None else 0
        got, pos = gvrs.pack_tile_records_multi(ctx, arenas, offsets, lens, base_pos, checksum, tile_index=tile_index,
                                                first_tile_index=first)
        want, want_pos = [], []
        at = base_pos
        for t in range(n):
            ti = first + t if tile_index is None else int(tile_index[t])
            rec = host_record(ti, [payloads[e][t] for e in range(n_elements)], oracle.crc32c if checksum else None)
            want.append(rec)
            want_pos.append(at + 8)
            at += len(rec)
        want = b"".join(want)
        assert got == want, (base_pos, checksum)
        assert [int(p) for p in pos] == want_pos
        if n_elements == 1:
            single, spos = gvrs.pack_tile_records(ctx, arenas[0], offsets[0], lens[0], base_pos, checksum, tile_index=tile_index,
                                                  first_tile_index=first)
            assert single == got and np.array_equal(spos, pos)
        if tile_index is None:
            batches = _device_batches(g4, torch, arenas, offsets, lens)
            drec, dpos = gvrs.pack_tile_records_multi_device(ctx, batches, base_pos, checksum, first_tile_index=first)
            torch.cuda.synchronize()
            assert drec.cpu().numpy().tobytes() == want
            assert [int(p) for p in dpos.cpu()] == want_pos
    # a record total above the capacity reports the size needed; argument checks
    L = _lib.lib()
    total = C.c_uint64(0)
    out = np.zeros(64, np.uint8)
    cp = np.zeros(n, np.uint64)
    ptr = lambda xs: (C.c_void_p * n_elements)(*[x.ctypes.data for x in xs])  # noqa: E731
    st = L.g4_pack_tile_records_multi(ctx._h, 0, n_elements, ptr(arenas), ptr(offsets), ptr(lens), None, 0, n, 0, 0, out.ctypes.data,
                                      64, cp.ctypes.data, C.byref(total))
    assert st == G4_ERR_CAPACITY
    assert total.value == len(want)
    for bad_e in (0, 65):
        st = L.g4_pack_tile_records_multi(ctx._h, 0, bad_e, ptr(arenas), ptr(offsets), ptr(lens), None, 0, n, 0, 0, out.ctypes.data,
                                          64, cp.ctypes.data, C.byref(total))
        assert st == G4_ERR_UNSUPPORTED
        st = L.g4_unpack_tile_records_multi(ctx._h, 0, bad_e, out.ctypes.data, 64, cp.ctypes.data, n, 0, out.ctypes.data,
                                            out.ctypes.data, out.ctypes.data)
        assert st == G4_ERR_UNSUPPORTED
    st = L.g4_pack_tile_records_multi(ctx._h, 0, n_elements, ptr(arenas), ptr(offsets), ptr(lens), None, 0, n, 0, 4, out.ctypes.data,
                                      64, cp.ctypes.data, C.byref(total))
    assert st == G4_ERR_ARG  # base_pos not a multiple of 8


@pytest.mark.gpu
@pytest.mark.parametrize("n_elements", [1, 2, 3, 5, 8])
def test_unpack_matches_host_walk_and_flags_damage(g4, oracle, n_elements):
    import torch

    from gridfour_b200 import gvrs

    ctx = g4.Context.default()
    rng = np.random.default_rng(200 + n_elements)
    n = 300
    arenas, offsets, lens, payloads = make_batch(rng, n_elements, n)
    base_pos = 1024
    recs, pos = gvrs.pack_tile_records_multi(ctx, arenas, offsets, lens, base_pos, True)
    image = bytes(base_pos) + recs  # ends exactly at the last record's end
    pos = pos.copy()
    pos[[5, 77, 200]] = 0  # absent tiles
    want_off, want_lens = host_walk(image, pos, n_elements)
    for checksum in (True, False):
        off, ln, st = gvrs.unpack_tile_records_multi(ctx, image, pos, n_elements, checksum)
        assert np.array_equal(off, want_off) and np.array_equal(ln, want_lens)
        assert [int(s) for s in st] == [G4_DECLINED if int(p) == 0 else G4_OK for p in pos]
        for e in range(n_elements):
            for t in (0, 1, 150, 298):
                assert image[int(off[e, t]):int(off[e, t]) + int(ln[e, t])] == payloads[e][t]
    if n_elements == 1:
        s_off, s_ln, s_st = gvrs.unpack_tile_records(ctx, image, pos, True)
        assert np.array_equal(s_off, off[0]) and np.array_equal(s_ln, ln[0]) and np.array_equal(s_st, st)
    # device form
    d_off, d_ln, d_st = gvrs.unpack_tile_records_multi_device(ctx, torch.frombuffer(bytearray(image), dtype=torch.uint8).cuda(),
                                                              torch.from_numpy(pos.astype(np.int64)).cuda(), n_elements, True)
    torch.cuda.synchronize()
    assert np.array_equal(d_off.cpu().numpy().astype(np.uint64), want_off)
    assert np.array_equal(d_ln.cpu().numpy().astype(np.uint32), want_lens) and np.array_equal(d_st.cpu().numpy(), st)

    def len_field(t, e):
        q = int(pos[t]) + 4
        for k in range(e):
            q += 4 + struct.unpack_from("<i", image, q)[0]
        return q

    def record_end(t):
        return int(pos[t]) - 8 + struct.unpack_from("<i", image, int(pos[t]) - 8)[0]

    last = n - 1  # its record ends the image
    assert record_end(last) == len(image)
    cases = []  # (tile, mutation of the image or None, replacement content position or None, status with / without checksum)
    for t in (40, last):
        rp = int(pos[t]) - 8
        cases += [(t, lambda b, rp=rp: b.__setitem__(rp + 4, 1), None, (G4_ERR_FORMAT,) * 2),
                  (t, lambda b, rp=rp: struct.pack_into("<i", b, rp, struct.unpack_from("<i", b, rp)[0] + 4), None, (G4_ERR_FORMAT,) * 2),
                  (t, None, int(pos[t]) + 4, (G4_ERR_FORMAT,) * 2),
                  (t, None, int(pos[t]) + 1, (G4_ERR_FORMAT,) * 2),
                  (t, None, (len(image) + 15) & ~7, (G4_ERR_FORMAT,) * 2),
                  (t, None, 1 << 40, (G4_ERR_FORMAT,) * 2)]
        if t == last:  # a size that runs one record size step past the end of the image
            cases.append((t, lambda b, rp=rp: struct.pack_into("<i", b, rp, struct.unpack_from("<i", b, rp)[0] + 8), None,
                          (G4_ERR_FORMAT,) * 2))
        for e in sorted({0, n_elements // 2, n_elements - 1}):
            q = len_field(t, e)
            room = record_end(t) - 4 - (q + 4)  # the longest len that still ends at or before the checksum field

            def past(b, q=q, room=room):
                struct.pack_into("<i", b, q, room + 1)

            def bit31(b, q=q):
                struct.pack_into("<I", b, q, struct.unpack_from("<I", b, q)[0] | 0x80000000)

            cases += [(t, past, None, (G4_ERR_FORMAT,) * 2), (t, bit31, None, (G4_ERR_FORMAT,) * 2)]
            if e == n_elements - 1 and room != struct.unpack_from("<i", image, q)[0]:
                # a chain that ends exactly at the checksum field is sound (its CRC no longer matches)
                cases.append((t, lambda b, q=q, room=room: struct.pack_into("<i", b, q, room), None, (G4_CHECKSUM_MISMATCH, G4_OK)))
            if int(lens[e][t]):
                cases.append((t, lambda b, q=q: b.__setitem__(q + 4, b[q + 4] ^ 0x20), None, (G4_CHECKSUM_MISMATCH, G4_OK)))
    for t, mutate, new_pos, expect in cases:
        b = bytearray(image)
        if mutate:
            mutate(b)
        p = pos.copy()
        if new_pos is not None:
            p[t] = new_pos
        for checksum, want_st in zip((True, False), expect):
            off, ln, st = gvrs.unpack_tile_records_multi(ctx, bytes(b), p, n_elements, checksum)
            assert int(st[t]) == want_st, (t, checksum, new_pos)
            others = np.arange(n) != t
            assert np.array_equal(st[others], [G4_DECLINED if int(x) == 0 else G4_OK for x in pos[others]])
            assert np.array_equal(off[:, others], want_off[:, others]) and np.array_equal(ln[:, others], want_lens[:, others])
            if want_st != G4_OK:
                assert not off[:, t].any() and not ln[:, t].any()


def _master_for(g4, codecs):
    spec = g4.CodecSpecification(default=False)
    classes = {"GvrsHuffman": (g4.CodecHuffman,), "GvrsDeflate": (g4.CodecDeflate,), "GvrsFloat": (g4.CodecFloat,),
               "GvrsCanonicalHuffman": (g4.CodecCanonHuffman,), "LSOP12": (g4.LsEncoder12, g4.LsDecoder12)}
    for c in codecs:
        spec.addCompressionCodec(c, *classes[c])
    return g4.CodecMaster(spec)


CODECS = ["GvrsHuffman", "GvrsDeflate", "GvrsFloat", "LSOP12"]


@pytest.fixture(scope="module")
def three_element_file(g4, oracle):
    """500 x 700 in 90 x 120 tiles: an integer element (fill -9999), a float element (NaN fill), a short element (fill -500)."""
    from gridfour_b200 import gvrs

    rows, cols = 500, 700
    z = oracle.terrain_i32(0, 0, rows, cols)
    z[100:130, 200:260] = -9999
    f = oracle.terrain_f32(500, 900, rows, cols)
    f[300:340, 10:50] = np.float32("nan")
    s = (oracle.terrain_i32(2000, 0, rows, cols) // 8).astype(np.int16)
    s[s == -500] = -499
    short = gvrs.ElementSpec(gvrs.ELEM_SHORT, "s", range_block=struct.pack("<hhh", -32767, 32767, -500))
    spec = gvrs.GvrsSpec(rows, cols, 90, 120, [gvrs.ElementSpec.integer("z", fill_value=-9999), gvrs.ElementSpec.floating("f"), short],
                         CODECS, checksum=True)
    master = _master_for(g4, CODECS)
    w = gvrs.GvrsWriter(spec, uuid=bytes(range(16)), time_modified=1700000000000)
    for name, rid, typ, content, desc in gvrs.codec_metadata(CODECS):
        w.add_metadata(name, rid, typ, content, desc)
    batches = w.add_rasters(master, [z, f, s])
    return w.finish(master._context()), [z, f, s], batches, master, spec


@pytest.mark.gpu
def test_three_element_raster_round_trip(g4, oracle, three_element_file):
    from gridfour_b200 import gvrs

    image, grids, batches, master, spec = three_element_file
    ctx = master._context()
    img = gvrs.GvrsImage.parse(image)
    assert img.verify_checksums(ctx) == len(img.records) + 1
    assert (spec.tiles_down, spec.tiles_across) == (6, 6)
    got = img.read_rasters(master, crop=True)
    for g, want in zip(got, grids):
        assert g.dtype == want.dtype and np.array_equal(g.view(np.uint8), np.ascontiguousarray(want).view(np.uint8))
    # every element payload is the oracle's packing of its tile (fill values in the margin of the edge tiles)
    ids = [ORACLE_IDS[c] for c in CODECS]
    tr, tc = spec.tile_rows, spec.tile_cols
    d = img.tile_directory()
    assert sorted(d) == list(range(36))
    n_unaligned = 0
    for k, (e, g) in enumerate(zip(spec.elements, grids)):
        full = np.full((6 * tr, 6 * tc), e.fill_value, dtype=g.dtype)
        full[:spec.n_rows, :spec.n_cols] = g
        std = e.standard_size(tr * tc)
        for t in range(36):
            r, c = divmod(t, 6)
            tile = np.ascontiguousarray(full[r * tr:(r + 1) * tr, c * tc:(c + 1) * tc])
            if e.type_code == gvrs.ELEM_FLOAT:
                want = oracle.master_encode_f32(ids, tile)
            elif e.type_code == gvrs.ELEM_SHORT:
                wide = tile.astype(np.int32)
                wide[tile == e.fill_value] = -(2 ** 31)
                want = oracle.master_encode_i32(ids, wide)
                if len(want) >= std or len(want) == 4 * tr * tc:
                    want = tile.astype("<i2").tobytes().ljust(std, b"\0")
            else:
                want = oracle.master_encode_i32(ids, tile)
            assert batches[k].payload(t) == want, (k, t)
            q = d[t] + 4
            for _ in range(k):
                q += 4 + struct.unpack_from("<i", image, q)[0]
            assert image[q + 4:q + 4 + len(want)] == want
            n_unaligned += (q + 4) % 4 != 0
    assert n_unaligned > 0  # payloads after the first one sit at any byte offset of the image
    for k in range(3):
        one = img.read_raster(master, element=k)
        assert np.array_equal(one.view(np.uint8), img.read_rasters(master)[k].view(np.uint8))
    # a flipped payload bit is caught by the record checksum
    bad = bytearray(image)
    q = d[20] + 4
    q += 4 + struct.unpack_from("<i", image, q)[0]
    bad[q + 4 + 10] ^= 0x04
    with pytest.raises(IOError, match="Checksum mismatch in a tile record"):
        gvrs.GvrsImage.parse(bytes(bad)).read_rasters(master)
    # a directory entry outside the image is a damaged record, not a struct.error
    bad = bytearray(image)
    img2 = gvrs.GvrsImage.parse(image)
    cell = img2.pos_tile_dir + 24 + 4 * 3  # tile 3 of the (non-extended) directory
    struct.pack_into("<I", bad, cell, (len(image) + 64) // 8)
    with pytest.raises(IOError, match="damaged tile record for tile 3"):
        gvrs.GvrsImage.parse(bytes(bad)).read_raster(master, element=1, verify=False)


@pytest.mark.gpu
def test_device_resident_read(g4, three_element_file):
    import torch

    from gridfour_b200 import gvrs

    image, grids, batches, master, spec = three_element_file
    img = gvrs.GvrsImage.parse(image)
    host = img.read_rasters(master)
    n = spec.tiles_down * spec.tiles_across
    pos = np.zeros(n, np.int64)
    for t, p in img.tile_directory().items():
        pos[t] = p
    dimg = torch.frombuffer(bytearray(image), dtype=torch.uint8).cuda()
    off, lens, st = gvrs.unpack_tile_records_multi_device(master._context(), dimg, torch.from_numpy(pos).cuda(), 3, True)
    torch.cuda.synchronize()
    assert int((st != 0).sum()) == 0
    for k, e in enumerate(spec.elements):
        dt = {gvrs.ELEM_INTEGER: np.int32, gvrs.ELEM_FLOAT: np.float32, gvrs.ELEM_SHORT: np.int16}[e.type_code]
        band = master._band((spec.tiles_down * spec.tile_rows, spec.tiles_across * spec.tile_cols), dt, spec.tile_rows, spec.tile_cols,
                            fillValue=e.fill_value if e.type_code == gvrs.ELEM_SHORT else None)
        out = master.decodeTiles(g4.TileBatch(dimg, off[k], lens[k], None, None, None, int(dimg.numel()), band))
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy().view(np.uint8), host[k].view(np.uint8)), k
