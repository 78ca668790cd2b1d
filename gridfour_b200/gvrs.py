"""GVRS file images either side of the codec path (SURVEY.md section 8f, row 1).

Host-side mirror of the reference's file layout -- pure offset arithmetic, no sample data is touched on the CPU:
  * C/gvrs/GvrsFile.java:241-300,560-623        preamble, header record, fixed header slots, close() sequence
  * C/gvrs/GvrsFileSpecification.java:1170-1285  specification block (write) and :960-1045 (read)
  * C/gvrs/RecordManager.java:70-78,137-139,161-204,386-490,835-883,991-1017   records, tile records, directories
  * C/gvrs/TileDirectory.java:244-278            tile directory (int32 = content position / 8)
  * C/gvrs/GvrsMetadata.java:217-234             metadata record content
  * C/io/BufferedRandomAccessFile.java:689-701   leWriteUTF = [length:uint16 LE][UTF-8 bytes]
(C/ = /root/reference/core/src/main/java/org/gridfour/).

Everything that walks sample bytes runs on the GPU through the C ABI: record checksums (g4_crc32c), tile-record framing
(g4_pack_tile_records), record validation + payload location (g4_unpack_tile_records) and the codecs themselves
(g4_encode_tiles / g4_decode_tiles with the file image as the arena).  Rasters with several elements per tile take the
same path: one g4_encode_tiles call per element, then g4_pack_tile_records_multi frames [tileIndex] and a [len][bytes]
pair per element into each record; g4_unpack_tile_records_multi validates the records and locates every element's payload
in one call, and each element is decoded straight from the image (GvrsWriter.add_rasters, GvrsImage.read_rasters).
add_tile_record_host frames one record on the host, for records whose size the caller dictates.
"""
import ctypes as C
import struct

import numpy as np

from . import _lib
from ._lib import G4_MEM_HOST, check

RECORD_FREESPACE, RECORD_METADATA, RECORD_TILE, RECORD_FREESPACE_DIR, RECORD_METADATA_DIR, RECORD_TILE_DIR, RECORD_HEADER = range(7)
ELEM_INTEGER, ELEM_INT_CODED_FLOAT, ELEM_FLOAT, ELEM_SHORT = 0, 1, 2, 3  # GvrsElementType.java:50-64
_ELEM_BYTES = {ELEM_INTEGER: 4, ELEM_INT_CODED_FLOAT: 4, ELEM_FLOAT: 4, ELEM_SHORT: 2}
_ELEM_DTYPE = {ELEM_INTEGER: np.int32, ELEM_INT_CODED_FLOAT: np.int32, ELEM_FLOAT: np.float32, ELEM_SHORT: np.int16}
FILEPOS_HEADER_RECORD = 16
FILEPOS_FREESPACE_DIR, FILEPOS_METADATA_DIR, FILEPOS_TILE_DIR = 56, 64, 80
METADATA_TYPE_STRING = 9  # GvrsMetadataType.STRING (the type byte of the two codec metadata records in every sample file)


def multiple_of_8(n):
    return (n + 7) & ~7


def _utf(s):
    b = (s or "").encode("utf-8")
    return struct.pack("<H", len(b)) + b


class _Reader:
    def __init__(self, b, pos):
        self.b, self.pos = b, pos

    def take(self, fmt):
        v = struct.unpack_from(fmt, self.b, self.pos)
        self.pos += struct.calcsize(fmt)
        return v if len(v) > 1 else v[0]

    def raw(self, n):
        v = bytes(self.b[self.pos:self.pos + n])
        self.pos += n
        return v

    def utf(self):
        n = self.take("<H")
        return self.raw(n).decode("utf-8")

    def skip_to_4(self):
        self.pos += (-self.pos) & 3


class ElementSpec:
    """GvrsElementSpecification*: type code, name, the type's range block (kept as raw little-endian bytes so that a
    re-serialised header is bit-identical), label, description, unit of measure."""

    def __init__(self, type_code, name, continuous=False, range_block=b"", label="", description="", unit=""):
        self.type_code, self.name, self.continuous = type_code, name, continuous
        self.range_block, self.label, self.description, self.unit = range_block, label, description, unit

    @property
    def fill_value(self):
        if self.type_code == ELEM_SHORT:
            return struct.unpack_from("<h", self.range_block, 4)[0]
        if self.type_code == ELEM_INTEGER:
            return struct.unpack_from("<i", self.range_block, 8)[0]
        if self.type_code == ELEM_FLOAT:
            return struct.unpack_from("<f", self.range_block, 8)[0]
        return struct.unpack_from("<i", self.range_block, 28)[0]  # INT_CODED_FLOAT: the integer fill value

    @staticmethod
    def integer(name, min_value=-(2 ** 31) + 1, max_value=2 ** 31 - 1, fill_value=-(2 ** 31), **kw):
        return ElementSpec(ELEM_INTEGER, name, range_block=struct.pack("<iii", min_value, max_value, fill_value), **kw)

    @staticmethod
    def floating(name, min_value=-3.4028235e38, max_value=3.4028235e38, fill_value=float("nan"), **kw):
        return ElementSpec(ELEM_FLOAT, name, range_block=struct.pack("<fff", min_value, max_value, fill_value), **kw)

    @staticmethod
    def int_coded_float(name, scale, offset=0.0, min_value=None, max_value=None, fill_value=float("nan"), **kw):
        """GvrsElementSpecificationIntCodedFloat.  The range block is [min f32][max f32][fill f32][scale f32][offset f32]
        [iMin][iMax][iFill]: with min and max given, the int bounds are their codes; without them, the int bounds are
        +-(2^31 - 1) and the float bounds are the values of those codes.  A NaN fill is coded as INT4_NULL_CODE.  (Header
        metadata computed with numpy float32 / float64 in the arithmetic of g4_icf_desc; sample data is mapped on the GPU.)"""
        f32 = np.float32
        scale, offset, fill = f32(scale), f32(offset), f32(fill_value)
        if not np.isfinite(scale) or scale == 0:
            raise ValueError("integer-coded float: the scale must be finite and not zero")

        def code(v):
            with np.errstate(invalid="ignore", over="ignore"):
                d = np.floor(np.float64((f32(v) - offset) * scale) + 0.5)
            return 0 if np.isnan(d) else int(min(max(d, -2.0 ** 31), 2.0 ** 31 - 1))

        def value(k):
            return (f32(k) / scale) + offset

        if (min_value is None) != (max_value is None):
            raise ValueError("integer-coded float: give both min_value and max_value, or neither")
        if min_value is None:
            i_min, i_max = -(2 ** 31) + 1, 2 ** 31 - 1
            min_value, max_value = value(i_min), value(i_max)
        else:
            i_min, i_max = code(min_value), code(max_value)
        i_fill = -(2 ** 31) if np.isnan(fill) else code(fill)
        block = np.array([min_value, max_value, fill, scale, offset], "<f4").tobytes() + struct.pack("<iii", i_min, i_max, i_fill)
        return ElementSpec(ELEM_INT_CODED_FLOAT, name, range_block=block, **kw)

    @property
    def icf(self):
        """The IntCodedFloat of an integer-coded float element (None for the other types)."""
        if self.type_code != ELEM_INT_CODED_FLOAT:
            return None
        from .codecs import IntCodedFloat

        fill, scale, offset = np.frombuffer(self.range_block, "<f4", 3, 8)
        return IntCodedFloat(scale, offset, struct.unpack_from("<i", self.range_block, 28)[0], fill)

    def standard_size(self, n_cells):
        n = n_cells * _ELEM_BYTES[self.type_code]
        return (n + 3) & ~3  # TileElement.java:89-93: the 2-byte form is padded to a multiple of 4


_RANGE_BYTES = {ELEM_SHORT: 6, ELEM_FLOAT: 12, ELEM_INT_CODED_FLOAT: 32, ELEM_INTEGER: 12}


class GvrsSpec:
    """The part of GvrsFileSpecification that is stored in the header.  The georeferencing block (raster space code,
    coordinate system code, 18 doubles) is opaque to the codec path and kept as raw bytes."""

    def __init__(self, n_rows, n_cols, tile_rows, tile_cols, elements, codecs=(), checksum=False, product_label="",
                 georef=None):
        self.n_rows, self.n_cols, self.tile_rows, self.tile_cols = n_rows, n_cols, tile_rows, tile_cols
        self.elements, self.codecs, self.checksum, self.product_label = list(elements), list(codecs), bool(checksum), product_label
        if georef is None:  # what GvrsFileSpecification's constructor sets up: unit cells, identity transforms
            d = [0.0, 0.0, n_cols - 1.0, n_rows - 1.0, 1.0, 1.0, 1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0, 0.0]
            georef = bytes([0, 0, 0, 0, 0, 0, 0]) + struct.pack("<18d", *d)
        self.georef = georef  # rasterSpace, coordinateSystem, 5 reserved bytes, 18 doubles = 151 bytes

    @property
    def tiles_down(self):
        return (self.n_rows + self.tile_rows - 1) // self.tile_rows

    @property
    def tiles_across(self):
        return (self.n_cols + self.tile_cols - 1) // self.tile_cols

    @property
    def standard_tile_bytes(self):
        n = self.tile_rows * self.tile_cols
        return sum(e.standard_size(n) for e in self.elements)

    def serialize(self, file_pos):
        """GvrsFileSpecification.write (:1170-1285); file_pos = absolute position of the first byte (padding to multiples
        of 4 is relative to the file position, padMultipleOf4 :1158-1164)."""
        out = bytearray()
        out += struct.pack("<iiiiii", self.n_rows, self.n_cols, self.tile_rows, self.tile_cols, 0, 0)
        out += bytes([1 if self.checksum else 0]) + self.georef
        out += struct.pack("<i", len(self.elements))
        for e in self.elements:
            out += bytes([e.type_code, 1 if e.continuous else 0]) + bytes(6) + _utf(e.name)
            out += bytes((-(file_pos + len(out))) & 3)
            out += e.range_block + _utf(e.label) + _utf(e.description) + _utf(e.unit)
            out += bytes((-(file_pos + len(out))) & 3)
        out += struct.pack("<i", len(self.codecs))
        for c in self.codecs:
            out += _utf(c)
        out += _utf(self.product_label)
        return bytes(out)

    @staticmethod
    def parse(b, pos):
        r = _Reader(b, pos)
        n_rows, n_cols, tile_rows, tile_cols, _, _ = r.take("<iiiiii")
        checksum = r.take("<B") != 0
        georef = r.raw(7 + 18 * 8)
        elements = []
        for _ in range(r.take("<i")):
            type_code, continuous = r.take("<BB")
            r.raw(6)
            name = r.utf()
            r.skip_to_4()
            if type_code not in _RANGE_BYTES:
                raise IOError("Unsupported value for data-type code: %d" % type_code)
            block = r.raw(_RANGE_BYTES[type_code])
            label, description, unit = r.utf(), r.utf(), r.utf()
            r.skip_to_4()
            elements.append(ElementSpec(type_code, name, continuous != 0, block, label, description, unit))
        codecs = [r.utf() for _ in range(r.take("<i"))]
        label = r.utf()
        return GvrsSpec(n_rows, n_cols, tile_rows, tile_cols, elements, codecs, checksum, label, georef), r.pos


class Record:
    def __init__(self, pos, size, type_code, body):
        self.pos, self.size, self.type_code, self.body = pos, size, type_code, body  # body = bytes 8 .. size-4 (content + padding)

    @property
    def content_pos(self):
        return self.pos + 8


class GvrsImage:
    """A parsed GVRS file image (version 1.3 and later).  `records` lists every record after the header in file order."""

    def __init__(self):
        self.version = (1, 4)
        self.uuid = bytes(16)
        self.time_modified = 0
        self.time_opened = 0
        self.spec = None
        self.records = []
        self.header_size = 0
        self.pos_freespace_dir = self.pos_metadata_dir = self.pos_tile_dir = 0
        self.image = b""

    # ---- reading ---------------------------------------------------------------------------------------------------
    @staticmethod
    def parse(image):
        b = bytes(image)
        if b[:11] != b"gvrs raster" or len(b) < 112:
            raise IOError("not a GVRS raster file")
        g = GvrsImage()
        g.image = b
        g.version = (b[12], b[13])
        if g.version < (1, 3):
            raise IOError("GVRS version %d.%d is not supported (1.3 and later)" % g.version)
        g.header_size, htype = struct.unpack_from("<iB", b, FILEPOS_HEADER_RECORD)
        if htype != RECORD_HEADER or g.header_size < 96 or FILEPOS_HEADER_RECORD + g.header_size > len(b):
            raise IOError("damaged GVRS header record")
        g.uuid = b[24:40]
        g.time_modified, g.time_opened = struct.unpack_from("<qq", b, 40)
        g.pos_freespace_dir, g.pos_metadata_dir = struct.unpack_from("<qq", b, FILEPOS_FREESPACE_DIR)
        g.pos_tile_dir = struct.unpack_from("<q", b, FILEPOS_TILE_DIR)[0]
        g.spec, _ = GvrsSpec.parse(b, 104)
        pos = FILEPOS_HEADER_RECORD + g.header_size
        while pos + 8 <= len(b):
            size, type_code = struct.unpack_from("<iB", b, pos)
            if size < 16 or (size & 7) or pos + size > len(b) or type_code > RECORD_TILE_DIR:
                raise IOError("damaged record at file position %d" % pos)
            g.records.append(Record(pos, size, type_code, b[pos + 8:pos + size - 4]))
            pos += size
        return g

    def tile_directory(self):
        """{tileIndex: content position}; RecordManager.readTileDirectory (:835-858) + TileDirectory.readTilePositions."""
        if self.pos_tile_dir == 0:
            return {}
        b, p = self.image, self.pos_tile_dir
        extended = b[p + 1] != 0
        row0, col0, n_rows, n_cols = struct.unpack_from("<iiii", b, p + 8)
        out = {}
        q = p + 24
        for i in range(n_rows):
            for j in range(n_cols):
                if extended:  # TileDirectoryExtended: 64-bit positions
                    off = struct.unpack_from("<q", b, q)[0]
                    q += 8
                else:
                    off = struct.unpack_from("<I", b, q)[0] * 8
                    q += 4
                if off:
                    out[(row0 + i) * self.spec.tiles_across + (col0 + j)] = off
        return out

    def record_ranges(self, include_header=True):
        """(offsets, sizes) of the checksummed part of every record: the first size-4 bytes."""
        recs = ([(FILEPOS_HEADER_RECORD, self.header_size)] if include_header else []) + [(r.pos, r.size) for r in self.records]
        return (np.array([p for p, _ in recs], dtype=np.uint64), np.array([s - 4 for _, s in recs], dtype=np.uint32),
                np.array([struct.unpack_from("<I", self.image, p + s - 4)[0] for p, s in recs], dtype=np.uint32))

    def verify_checksums(self, context):
        """GPU CRC-32C of every record against the stored values.  Returns the number of records checked."""
        if not self.spec.checksum:
            return 0
        off, size, stored = self.record_ranges()
        crc = crc32c_ranges(context, self.image, off, size)
        bad = np.nonzero(crc != stored)[0]
        if len(bad):
            raise IOError("Checksum mismatch in record at file position %d" % int(off[bad[0]]))
        return len(off)

    def _locate_all(self, ctx, verify):
        """(payload offsets [E, n], lengths [E, n], status [n]) of every element of every tile, in one GPU call; raises
        IOError for a damaged tile record or, with verify, a record whose checksum differs."""
        from ._lib import G4_CHECKSUM_MISMATCH

        spec = self.spec
        n_tiles = spec.tiles_down * spec.tiles_across
        pos = np.zeros(n_tiles, dtype=np.uint64)
        for t, p in self.tile_directory().items():
            pos[t] = p
        checksum = verify and spec.checksum
        if len(spec.elements) == 1:
            payload_off, lens, status = unpack_tile_records(ctx, self.image, pos, checksum=checksum)
            payload_off, lens = payload_off[None], lens[None]
        else:
            payload_off, lens, status = unpack_tile_records_multi(ctx, self.image, pos, len(spec.elements), checksum=checksum)
        bad = np.nonzero(status < 0)[0]
        if len(bad):
            raise IOError("damaged tile record for tile %d" % int(bad[0]))
        if np.any(status == G4_CHECKSUM_MISMATCH):
            raise IOError("Checksum mismatch in a tile record")
        return payload_off, lens, status

    def locate_payloads(self, ctx, element=0, verify=True):
        """(payload offsets, lengths, status) of one element of every tile, as g4_decode_tiles takes them with the file image
        as its arena; status G4_DECLINED marks tiles the file does not hold.  The records are validated, their checksums
        checked and their payloads located on the GPU (g4_unpack_tile_records, or g4_unpack_tile_records_multi for rasters
        with several elements per tile)."""
        if not 0 <= element < len(self.spec.elements):
            raise ValueError("no such element")
        payload_off, lens, status = self._locate_all(ctx, verify)
        return payload_off[element], lens[element], status

    def _decode_element(self, master, element, payload_off, lens, status, crop, as_float):
        spec = self.spec
        e = spec.elements[element]
        grid = master.decodeImageTiles(self.image, payload_off, lens, status, spec.tiles_down, spec.tiles_across, spec.tile_rows,
                                       spec.tile_cols, _ELEM_DTYPE[e.type_code], e.fill_value, icf=e.icf if as_float else None)
        return grid[:spec.n_rows, :spec.n_cols] if crop else grid

    def read_raster(self, master, element=0, verify=True, crop=False, as_float=False):
        """crop=True returns the n_rows x n_cols raster without the fill-valued margin of the edge tiles.
        Decodes every tile of one element of the raster on the GPU straight from the file image: the image is the arena
        of g4_decode_tiles; locate_payloads finds the payloads.  Tiles that are absent from the file come back filled with
        the element's fill value (RasterTile.setToNullState).  An integer-coded float element comes back as its int codes,
        or with as_float=True as float32 values (g4_decode_tiles_icf); as_float changes nothing for the other types."""
        payload_off, lens, status = self.locate_payloads(master._context(), element, verify)
        return self._decode_element(master, element, payload_off, lens, status, crop, as_float)

    def read_rasters(self, master, verify=True, crop=False, as_float=False):
        """Every element's raster, in specification order, from one validation + location call (read_raster per element
        would repeat it)."""
        payload_off, lens, status = self._locate_all(master._context(), verify)
        return [self._decode_element(master, k, payload_off[k], lens[k], status, crop, as_float) for k in range(len(self.spec.elements))]

    def to_device(self, context=None, device=None, verify=True):
        """The image resident on a GPU, for reads that leave their results there (GvrsDeviceImage).  Uploads the image
        once, then validates every tile record and locates every element's payloads on the device; raises IOError for a
        damaged tile record or, with verify, a record whose checksum differs, as read_raster does."""
        import warnings

        import torch

        from ._lib import G4_CHECKSUM_MISMATCH
        from .codecs import Context

        if device is None:
            device = context.device if context is not None else torch.cuda.current_device()
        dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        ctx = context or Context.default(dev.index)
        spec = self.spec
        n_tiles = spec.tiles_down * spec.tiles_across
        n = len(self.image)
        buf = torch.empty(multiple_of_8(n) + 8, dtype=torch.uint8, device=dev)  # the unpack calls take an 8-byte aligned image
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)  # the bytes are only read: torch warns about any read-only buffer
            host = torch.from_numpy(np.frombuffer(self.image, dtype=np.uint8))
        buf[:n].copy_(host)
        image = buf[:n]
        pos = np.zeros(n_tiles, dtype=np.int64)
        for t, p in self.tile_directory().items():
            pos[t] = p
        content_pos = torch.from_numpy(pos).to(dev)
        checksum = verify and spec.checksum
        ctx.after_torch_stream(dev)
        if len(spec.elements) == 1:
            payload_off, lens, status = unpack_tile_records_device(ctx, image, content_pos, checksum)
            payload_off, lens = payload_off[None], lens[None]
        else:
            payload_off, lens, status = unpack_tile_records_multi_device(ctx, image, content_pos, len(spec.elements), checksum)
        ctx.before_torch_stream(dev)
        st = status.cpu().numpy()
        bad = np.nonzero(st < 0)[0]
        if len(bad):
            raise IOError("damaged tile record for tile %d" % int(bad[0]))
        if np.any(st == G4_CHECKSUM_MISMATCH):
            raise IOError("Checksum mismatch in a tile record")
        return GvrsDeviceImage(self, image, payload_off, lens, status, ctx)


class GvrsDeviceImage:
    """A GVRS file image resident in device memory with its payloads located (GvrsImage.to_device).  Reads decode only the
    tiles a request touches, straight from the resident image, and return torch CUDA tensors (g4_decode_window):
    per read, nothing crosses PCIe but the status of the tiles read.  The reads run on the context the image was made
    with; `master` gives the codec list."""

    def __init__(self, host, image, payload_off, lens, status, context):
        self.host, self.spec = host, host.spec
        self.image, self.payload_off, self.lens, self.status = image, payload_off, lens, status  # [n] / [E, n] / [E, n] / [n]
        self.context = context
        self.device = image.device
        self.lastStatus = None  # per covering tile of the latest read, window-tile order (device tensor)

    def _element(self, element):
        if not 0 <= element < len(self.spec.elements):
            raise ValueError("no such element")
        return self.spec.elements[element]

    def read_block(self, master, row, col, n_rows, n_cols, element=0, as_float=False, out=None):
        """GvrsElement.readBlock: the n_rows x n_cols cells from (row, col), which must lie inside the raster (ValueError
        otherwise).  Returns a CUDA tensor: int32 for integer elements and the codes of integer-coded float elements,
        float32 for float elements and, with as_float, for integer-coded float values, int16 for short elements.  Tiles
        absent from the file read as the element's fill value.  `out` may be any 2-D CUDA tensor of that dtype and shape
        whose rows are contiguous, e.g. a slice of a larger mosaic; its other cells are left as they are."""
        spec = self.spec
        self._element(element)
        if row < 0 or col < 0 or row + n_rows > spec.n_rows or col + n_cols > spec.n_cols or n_rows < 1 or n_cols < 1:
            raise ValueError("block outside the raster")
        return self._read(master, row, col, n_rows, n_cols, element, as_float, out)

    def read_raster(self, master, element=0, crop=False, as_float=False):
        """The values GvrsImage.read_raster returns, as a CUDA tensor: the whole tile grid, or with crop the n_rows x n_cols
        raster."""
        spec = self.spec
        self._element(element)
        if crop:
            return self._read(master, 0, 0, spec.n_rows, spec.n_cols, element, as_float, None)
        return self._read(master, 0, 0, spec.tiles_down * spec.tile_rows, spec.tiles_across * spec.tile_cols, element, as_float, None)

    def _read(self, master, row, col, n_rows, n_cols, element, as_float, out):
        import torch

        from ._lib import G4_ELEM_F32, G4_ELEM_I16, G4_ELEM_I32, G4_ELEM_ICF, BandDesc

        spec = self.spec
        e = spec.elements[element]
        icf = e.icf if as_float else None
        band = BandDesc()
        band.tile_rows, band.tile_cols = spec.tile_rows, spec.tile_cols
        band.tiles_down, band.tiles_across = spec.tiles_down, spec.tiles_across
        band.grid_pitch = spec.tiles_across * spec.tile_cols
        if icf is not None:
            band.elem_type, dtype = G4_ELEM_ICF, torch.float32
            fill = struct.unpack("<I", bytes(C.c_float(float(icf.fill_value))))[0]  # the float g4_icf_desc carries
        elif e.type_code == ELEM_FLOAT:
            band.elem_type, dtype = G4_ELEM_F32, torch.float32
            fill = int(np.float32(e.fill_value).view(np.uint32))
        elif e.type_code == ELEM_SHORT:
            band.elem_type, dtype = G4_ELEM_I16, torch.int16
            fill = e.fill_value & 0xffff
        else:
            band.elem_type, dtype = G4_ELEM_I32, torch.int32
            fill = e.fill_value & 0xffffffff
        if out is None:
            out = torch.empty((n_rows, n_cols), dtype=dtype, device=self.device)
        elif not (isinstance(out, torch.Tensor) and out.device == self.device and out.dtype == dtype and out.dim() == 2
                  and tuple(out.shape) == (n_rows, n_cols) and (n_rows == 1 or out.stride(0) >= n_cols) and (n_cols == 1 or out.stride(1) == 1)):
            raise ValueError("out: a 2-D %s tensor of shape (%d, %d) on %s with contiguous rows" % (dtype, n_rows, n_cols, self.device))
        pitch = out.stride(0) if n_rows > 1 else n_cols
        t_down = (row + n_rows - 1) // spec.tile_rows - row // spec.tile_rows + 1
        t_across = (col + n_cols - 1) // spec.tile_cols - col // spec.tile_cols + 1
        status = torch.empty(t_down * t_across, dtype=torch.int32, device=self.device)
        d = icf.desc() if icf is not None else None
        ctx = self.context
        ctx.after_torch_stream(self.device)  # `out` may still be in use on torch's stream
        st = _lib.lib().g4_decode_window(ctx._h, C.byref(master._native_list()), C.byref(band), None if d is None else C.byref(d),
                                         self.image.data_ptr(), int(self.image.numel()), self.payload_off[element].data_ptr(),
                                         self.lens[element].data_ptr(), self.status.data_ptr(), fill, int(row), int(col), int(n_rows),
                                         int(n_cols), out.data_ptr(), int(pitch), status.data_ptr())
        ctx.before_torch_stream(self.device)
        self.lastStatus = status
        check(st, "g4_decode_window")
        return out


# ---- GPU-backed primitives -------------------------------------------------------------------------------------------
def _u8(buf):
    a = np.frombuffer(buf, dtype=np.uint8) if not isinstance(buf, np.ndarray) else buf
    return np.ascontiguousarray(a)


def crc32c_ranges(context, data, offsets, sizes):
    """CRC-32C (GridfourCRC32C) of data[offsets[i] : offsets[i]+sizes[i]] for every i, computed on the GPU."""
    a = _u8(data)
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    sz = np.ascontiguousarray(sizes, dtype=np.uint32)
    out = np.zeros(len(off), dtype=np.uint32)
    if len(off) and int((off + sz).max()) > a.size:
        raise ValueError("range outside the buffer")
    check(_lib.lib().g4_crc32c(context._h, G4_MEM_HOST, a.ctypes.data, off.ctypes.data, sz.ctypes.data, len(off), out.ctypes.data),
          "g4_crc32c")
    return out


def crc32c(context, data):
    return int(crc32c_ranges(context, data, [0], [len(data)])[0])


def pack_tile_records(context, arena, offsets, lens, base_pos, checksum, tile_index=None, first_tile_index=0):
    """RecordManager.writeTile framing of a batch of one-element tile payloads.  Returns (record bytes, content positions)."""
    a = _u8(arena)
    off = np.ascontiguousarray(offsets, dtype=np.uint64)
    ln = np.ascontiguousarray(lens, dtype=np.uint32)
    n = len(off)
    L = _lib.lib()
    cap = int(L.g4_tile_records_bound(n, int(ln.sum())))
    out = np.zeros(cap + 16, dtype=np.uint8)
    pos = np.zeros(n, dtype=np.uint64)
    total = C.c_uint64(0)
    idx = None if tile_index is None else np.ascontiguousarray(tile_index, dtype=np.int32)
    check(L.g4_pack_tile_records(context._h, G4_MEM_HOST, a.ctypes.data, off.ctypes.data, ln.ctypes.data,
                                 None if idx is None else idx.ctypes.data, int(first_tile_index), n, 1 if checksum else 0, int(base_pos),
                                 out.ctypes.data, cap, pos.ctypes.data, C.byref(total)), "g4_pack_tile_records")
    return out[:total.value].tobytes(), pos


def unpack_tile_records(context, image, content_pos, checksum):
    a = _u8(image)
    pos = np.ascontiguousarray(content_pos, dtype=np.uint64)
    n = len(pos)
    payload = np.zeros(n, dtype=np.uint64)
    lens = np.zeros(n, dtype=np.uint32)
    status = np.zeros(n, dtype=np.int32)
    check(_lib.lib().g4_unpack_tile_records(context._h, G4_MEM_HOST, a.ctypes.data, a.size, pos.ctypes.data, n, 1 if checksum else 0,
                                            payload.ctypes.data, lens.ctypes.data, status.ctypes.data), "g4_unpack_tile_records")
    return payload, lens, status


def pack_tile_records_device(context, batch, base_pos, checksum, first_tile_index=0):
    """Device-resident form: `batch` is the TileBatch of CodecMaster.encodeTiles on a CUDA tensor.  Returns (records,
    content positions) as torch CUDA tensors; nothing crosses PCIe except the 8-byte total."""
    import torch

    from ._lib import G4_MEM_DEVICE

    L = _lib.lib()
    n = int(batch.lens.numel())
    cap = int(L.g4_tile_records_bound(n, int(batch.total_bytes)))
    dev = batch.arena.device
    out = torch.empty(cap + 16, dtype=torch.uint8, device=dev)
    pos = torch.empty(n, dtype=torch.int64, device=dev)
    total = C.c_uint64(0)
    check(L.g4_pack_tile_records(context._h, G4_MEM_DEVICE, batch.arena.data_ptr(), batch.offsets.data_ptr(), batch.lens.data_ptr(), None,
                                 int(first_tile_index), n, 1 if checksum else 0, int(base_pos), out.data_ptr(), cap, pos.data_ptr(),
                                 C.byref(total)), "g4_pack_tile_records")
    return out[:total.value], pos


def unpack_tile_records_device(context, image, content_pos, checksum):
    """Device-resident form of unpack_tile_records: image and content_pos are torch CUDA tensors (uint8 / int64)."""
    import torch

    from ._lib import G4_MEM_DEVICE

    n = int(content_pos.numel())
    dev = image.device
    payload = torch.empty(n, dtype=torch.int64, device=dev)
    lens = torch.empty(n, dtype=torch.int32, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    check(_lib.lib().g4_unpack_tile_records(context._h, G4_MEM_DEVICE, image.data_ptr(), int(image.numel()), content_pos.data_ptr(), n,
                                            1 if checksum else 0, payload.data_ptr(), lens.data_ptr(), status.data_ptr()),
          "g4_unpack_tile_records")
    return payload, lens, status


def _pointers(buffers):
    return (C.c_void_p * len(buffers))(*buffers)


def pack_tile_records_multi(context, arenas, offsets, lens, base_pos, checksum, tile_index=None, first_tile_index=0):
    """RecordManager.writeTile framing of a batch of tiles with len(arenas) elements: element e of tile t is
    arenas[e][offsets[e][t] : + lens[e][t]].  Returns (record bytes, content positions)."""
    a = [_u8(x) for x in arenas]
    off = [np.ascontiguousarray(o, dtype=np.uint64) for o in offsets]
    ln = [np.ascontiguousarray(x, dtype=np.uint32) for x in lens]
    n = len(off[0]) if off else 0
    if len(off) != len(a) or len(ln) != len(a) or any(len(o) != n for o in off) or any(len(x) != n for x in ln):
        raise ValueError("pack_tile_records_multi: one offset and one length array of the same length per arena")
    L = _lib.lib()
    cap = int(L.g4_tile_records_bound_multi(n, len(a), sum(int(x.sum()) for x in ln)))
    out = np.zeros(cap + 16, dtype=np.uint8)
    pos = np.zeros(n, dtype=np.uint64)
    total = C.c_uint64(0)
    idx = None if tile_index is None else np.ascontiguousarray(tile_index, dtype=np.int32)
    check(L.g4_pack_tile_records_multi(context._h, G4_MEM_HOST, len(a), _pointers([x.ctypes.data for x in a]),
                                       _pointers([x.ctypes.data for x in off]), _pointers([x.ctypes.data for x in ln]),
                                       None if idx is None else idx.ctypes.data, int(first_tile_index), n, 1 if checksum else 0,
                                       int(base_pos), out.ctypes.data, cap, pos.ctypes.data, C.byref(total)), "g4_pack_tile_records_multi")
    return out[:total.value].tobytes(), pos


def unpack_tile_records_multi(context, image, content_pos, n_elements, checksum):
    """Inverse of pack_tile_records_multi.  Returns (payload offsets [E, n], lengths [E, n], status [n]); row e is what
    g4_decode_tiles takes for element e with the image as its arena."""
    a = _u8(image)
    pos = np.ascontiguousarray(content_pos, dtype=np.uint64)
    n = len(pos)
    payload = np.zeros((n_elements, n), dtype=np.uint64)
    lens = np.zeros((n_elements, n), dtype=np.uint32)
    status = np.zeros(n, dtype=np.int32)
    check(_lib.lib().g4_unpack_tile_records_multi(context._h, G4_MEM_HOST, int(n_elements), a.ctypes.data, a.size, pos.ctypes.data, n,
                                                  1 if checksum else 0, payload.ctypes.data, lens.ctypes.data, status.ctypes.data),
          "g4_unpack_tile_records_multi")
    return payload, lens, status


def pack_tile_records_multi_device(context, batches, base_pos, checksum, first_tile_index=0):
    """Device-resident form: `batches` holds one TileBatch of CodecMaster.encodeTiles on a CUDA tensor per element, all of
    the same tiles.  Returns (records, content positions) as torch CUDA tensors; nothing crosses PCIe except the 8-byte
    total."""
    import torch

    from ._lib import G4_MEM_DEVICE

    L = _lib.lib()
    n = int(batches[0].lens.numel()) if batches else 0
    if any(int(b.lens.numel()) != n for b in batches):
        raise ValueError("pack_tile_records_multi_device: every element's batch holds the same tiles")
    cap = int(L.g4_tile_records_bound_multi(n, len(batches), sum(int(b.total_bytes) for b in batches)))
    dev = batches[0].arena.device if batches else None
    out = torch.empty(cap + 16, dtype=torch.uint8, device=dev)
    pos = torch.empty(n, dtype=torch.int64, device=dev)
    total = C.c_uint64(0)
    check(L.g4_pack_tile_records_multi(context._h, G4_MEM_DEVICE, len(batches), _pointers([b.arena.data_ptr() for b in batches]),
                                       _pointers([b.offsets.data_ptr() for b in batches]), _pointers([b.lens.data_ptr() for b in batches]),
                                       None, int(first_tile_index), n, 1 if checksum else 0, int(base_pos), out.data_ptr(), cap,
                                       pos.data_ptr(), C.byref(total)), "g4_pack_tile_records_multi")
    return out[:total.value], pos


def unpack_tile_records_multi_device(context, image, content_pos, n_elements, checksum):
    """Device-resident form of unpack_tile_records_multi: image and content_pos are torch CUDA tensors (uint8 / int64).
    Returns [E, n] int64 offsets, [E, n] int32 lengths and [n] int32 status on the device."""
    import torch

    from ._lib import G4_MEM_DEVICE

    n = int(content_pos.numel())
    dev = image.device
    payload = torch.empty((n_elements, n), dtype=torch.int64, device=dev)
    lens = torch.empty((n_elements, n), dtype=torch.int32, device=dev)
    status = torch.empty(n, dtype=torch.int32, device=dev)
    check(_lib.lib().g4_unpack_tile_records_multi(context._h, G4_MEM_DEVICE, int(n_elements), image.data_ptr(), int(image.numel()),
                                                  content_pos.data_ptr(), n, 1 if checksum else 0, payload.data_ptr(), lens.data_ptr(),
                                                  status.data_ptr()), "g4_unpack_tile_records_multi")
    return payload, lens, status


# ---- writing ---------------------------------------------------------------------------------------------------------
def frame_record(type_code, content, size=None):
    """[size][type][0,0,0] content, zero padding, checksum field left zero (fileSpaceInitRecord / FinishRecord)."""
    if size is None:
        size = multiple_of_8(len(content) + 12)
    return struct.pack("<iB3x", size, type_code) + bytes(content) + bytes(size - 8 - len(content))


def metadata_content(name, record_id, type_code, content, description=""):
    """GvrsMetadata.write (:217-234)."""
    return _utf(name) + struct.pack("<iB3xi", record_id, type_code, len(content)) + bytes(content) + _utf(description)


def codec_metadata(codecs, java_classes=None):
    """The two records GvrsFile writes for a compressed file (GvrsFile.java:301-319): the Java class names per codec id
    ("GvrsJavaCodecs") and the id list ("GvrsCompressionCodecs")."""
    std = {
        "GvrsHuffman": ("org.gridfour.compress.CodecHuffman", "org.gridfour.compress.CodecHuffman"),
        "GvrsDeflate": ("org.gridfour.compress.CodecDeflate", "org.gridfour.compress.CodecDeflate"),
        "GvrsFloat": ("org.gridfour.compress.CodecFloat", "org.gridfour.compress.CodecFloat"),
        "GvrsCanonicalHuffman": ("org.gridfour.compress.canonicalHuffman.CodecCanonHuffman",) * 2,
        "LSOP12": ("org.gridfour.lsop.LsEncoder12", "org.gridfour.lsop.LsDecoder12"),
    }
    std.update(java_classes or {})
    java = "".join("%s,%s,%s\n" % (c, std[c][0], std[c][1]) for c in codecs).encode("utf-8")
    ids = "|".join(codecs).encode("utf-8")
    return [("GvrsJavaCodecs", 0, METADATA_TYPE_STRING, struct.pack("<i", len(java)) + java, "Class paths for Java compressors"),
            ("GvrsCompressionCodecs", 0, METADATA_TYPE_STRING, struct.pack("<i", len(ids)) + ids, "Compession codecs")]


def tile_directory_content(spec, positions, extended=False):
    """RecordManager.writeTileDirectory (:864-883) + TileDirectory.writeTilePositions (:266-278): the bounding box of the
    populated tiles, content position / 8 per cell."""
    cells = {}
    for t, p in positions.items():
        if p:
            cells[divmod(int(t), spec.tiles_across)] = int(p)
    out = bytearray([0, 1 if extended else 0, 0, 0, 0, 0, 0, 0])
    if not cells:
        return bytes(out + struct.pack("<iiii", 0, 0, 0, 0))
    rows, cols = [r for r, _ in cells], [c for _, c in cells]
    row0, col0, n_rows, n_cols = min(rows), min(cols), max(rows) - min(rows) + 1, max(cols) - min(cols) + 1
    out += struct.pack("<iiii", row0, col0, n_rows, n_cols)
    for i in range(n_rows):
        for j in range(n_cols):
            p = cells.get((row0 + i, col0 + j), 0)
            out += struct.pack("<q", p) if extended else struct.pack("<I", (p // 8) & 0xffffffff)
    return bytes(out)


def metadata_directory_content(entries):
    """RecordManager.writeMetadataDirectory (:991-1017); entries = (content position, name, record id, type code), in
    order of file position."""
    out = bytearray(struct.pack("<i", len(entries)))
    for pos, name, record_id, type_code in entries:
        out += struct.pack("<q", pos) + _utf(name) + struct.pack("<iB", record_id, type_code)
    return bytes(out)


class GvrsWriter:
    """Assembles a GVRS file image: header, records in the order they are added, directories, checksums.  Mirrors the
    sequence GvrsFile(File, spec) ... close() produces (GvrsFile.java:241-300, 560-623)."""

    def __init__(self, spec, uuid=None, time_modified=0, version=(1, 4)):
        self.spec, self.version = spec, version
        self.uuid = uuid if uuid is not None else bytes(16)
        self.time_modified = time_modified
        head = bytearray(b"gvrs raster".ljust(12, b"\0") + bytes([version[0], version[1], 0, 0]))
        head += struct.pack("<iB3x", 0, RECORD_HEADER) + self.uuid + struct.pack("<qq", time_modified, 0)
        head += struct.pack("<qq", 0, 0) + struct.pack("<H6x", 1) + struct.pack("<q", 0) + bytes(16)
        head += spec.serialize(len(head)) + bytes(8)
        content_pos = (len(head) + 4 + 7) & ~7
        head += bytes(content_pos - len(head))
        struct.pack_into("<i", head, FILEPOS_HEADER_RECORD, content_pos - FILEPOS_HEADER_RECORD)
        self.buf = head
        self.header_size = content_pos - FILEPOS_HEADER_RECORD
        self.record_spans = [(FILEPOS_HEADER_RECORD, self.header_size)]
        self.metadata_entries = []
        self.tile_positions = {}

    @property
    def file_pos(self):
        return len(self.buf)

    def add_record(self, type_code, content, size=None):
        pos = len(self.buf)
        rec = frame_record(type_code, content, size)
        self.buf += rec
        self.record_spans.append((pos, len(rec)))
        return pos + 8

    def add_metadata(self, name, record_id, type_code, content, description="", size=None):
        pos = self.add_record(RECORD_METADATA, metadata_content(name, record_id, type_code, content, description), size)
        self.metadata_entries.append((pos, name, record_id, type_code))
        return pos

    def add_tile_records(self, context, arena, offsets, lens, tile_index=None, first_tile_index=0):
        """Tile records of a batch, framed (and checksummed) on the GPU."""
        base = len(self.buf)
        recs, pos = pack_tile_records(context, arena, offsets, lens, base, self.spec.checksum, tile_index, first_tile_index)
        self.buf += recs
        idx = range(first_tile_index, first_tile_index + len(pos)) if tile_index is None else tile_index
        for t, p in zip(idx, pos):
            self.tile_positions[int(t)] = int(p)
        return pos

    def add_tile_records_multi(self, context, arenas, offsets, lens, tile_index=None, first_tile_index=0):
        """Tile records of a batch with one arena per element (pack_tile_records_multi), framed and checksummed on the GPU."""
        base = len(self.buf)
        recs, pos = pack_tile_records_multi(context, arenas, offsets, lens, base, self.spec.checksum, tile_index, first_tile_index)
        self.buf += recs
        idx = range(first_tile_index, first_tile_index + len(pos)) if tile_index is None else tile_index
        for t, p in zip(idx, pos):
            self.tile_positions[int(t)] = int(p)
        return pos

    def _encode_element(self, master, e, grid):
        """encodeTiles of one element's raster (numpy, n_rows x n_cols): the cells of the edge tiles that lie outside the
        raster hold the element's fill value, as a RasterTile that was never written there does (TileElementInt/Float/Short
        constructors fill the tile).  A float32 raster of an integer-coded float element holds values, which are mapped to
        codes on the GPU (the margin is filled with the float fill value first); an int32 raster holds the codes."""
        spec = self.spec
        shape = (spec.tiles_down * spec.tile_rows, spec.tiles_across * spec.tile_cols)
        if e.type_code == ELEM_INT_CODED_FLOAT and np.asarray(grid).dtype == np.float32:
            icf = e.icf
            full = np.full(shape, icf.fill_value, dtype=np.float32)
            full[:spec.n_rows, :spec.n_cols] = grid
            return master.encodeTiles(full, spec.tile_rows, spec.tile_cols, icf=icf)
        full = np.full(shape, e.fill_value, dtype=_ELEM_DTYPE[e.type_code])
        full[:spec.n_rows, :spec.n_cols] = grid
        return master.encodeTiles(full, spec.tile_rows, spec.tile_cols, fillValue=e.fill_value if e.type_code == ELEM_SHORT else None)

    def add_raster(self, master, grid):
        """A whole one-element raster (numpy, n_rows x n_cols): encodeTiles on the GPU, then the tile records.  Returns the
        TileBatch.  For an integer-coded float element, a float32 raster holds values and an int32 raster holds codes."""
        spec = self.spec
        if len(spec.elements) != 1 or grid.shape != (spec.n_rows, spec.n_cols):
            raise ValueError("add_raster: a one-element raster of the specified dimensions")
        batch = self._encode_element(master, spec.elements[0], grid)
        self.add_tile_records(master._context(), batch.arena, batch.offsets, batch.lens)
        return batch

    def add_rasters(self, master, grids):
        """Every element of a raster: grids[k] (numpy, n_rows x n_cols) is element k in specification order -- int32 for
        integer elements, float32 for float elements, int16 for short elements, and for integer-coded float elements float32
        values or int32 codes.  One encodeTiles per element, then one multi-element framing call.  Returns the TileBatch of
        every element."""
        spec = self.spec
        if len(grids) != len(spec.elements) or any(np.shape(g) != (spec.n_rows, spec.n_cols) for g in grids):
            raise ValueError("add_rasters: one raster of the specified dimensions per element")
        batches = [self._encode_element(master, e, g) for e, g in zip(spec.elements, grids)]
        self.add_tile_records_multi(master._context(), [b.arena for b in batches], [b.offsets for b in batches],
                                    [b.lens for b in batches])
        return batches

    def add_tile_record_host(self, tile_index, element_payloads, size=None):
        """One tile record with any number of elements, framed on the host: [tileIndex] then [len][bytes] per element;
        `size` may make the record larger than the content needs (as a reused file region leaves it)."""
        content = struct.pack("<i", tile_index) + b"".join(struct.pack("<i", len(p)) + bytes(p) for p in element_payloads)
        pos = self.add_record(RECORD_TILE, content, size)
        self.tile_positions[int(tile_index)] = pos
        return pos

    def finish(self, context, extended_directory=False, directory_order=("metadata", "tile")):
        """close(): metadata directory, tile directory, header slots, then every checksum -- all CRCs in one GPU call.
        (context=None leaves the checksum fields of the host-framed records zero: layout-only use in the CPU tests.)"""
        md_pos = td_pos = 0
        for which in directory_order:
            if which == "metadata" and self.metadata_entries:
                md_pos = self.add_record(RECORD_METADATA_DIR, metadata_directory_content(sorted(self.metadata_entries)))
            elif which == "tile":
                td_pos = self.add_record(RECORD_TILE_DIR, tile_directory_content(self.spec, self.tile_positions, extended_directory))
        struct.pack_into("<qq", self.buf, FILEPOS_FREESPACE_DIR, 0, md_pos)
        struct.pack_into("<q", self.buf, FILEPOS_TILE_DIR, td_pos)
        if self.spec.checksum and context is not None:
            off = np.array([p for p, _ in self.record_spans], dtype=np.uint64)
            size = np.array([s - 4 for _, s in self.record_spans], dtype=np.uint32)
            crc = crc32c_ranges(context, self.buf, off, size)
            for (p, s), c in zip(self.record_spans, crc):
                struct.pack_into("<I", self.buf, p + s - 4, int(c))
        return bytes(self.buf)
