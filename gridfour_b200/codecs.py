"""Host-side mirror of the reference's codec plugin API (same names, argument meaning and error behaviour).

Reference (paths under /root/reference/core/src/main/java/org/gridfour/):
  compress/ICompressionEncoder.java:46-92, compress/ICompressionDecoder.java:49-107
  gvrs/GvrsFileSpecification.java:221-230,1535-1724 (codec registration), gvrs/CodecMaster.java:142-203
  gvrs/TileElementInt.java:196-219 (raw fallback)
Everything that touches sample data is a call into libg4codec.so (CUDA); nothing is computed in Python.
"""
import ctypes as C
import threading

import numpy as np

from . import _lib
from ._lib import (G4_CODEC_CANON_HUFFMAN, G4_CODEC_DEFLATE, G4_CODEC_FLOAT, G4_CODEC_HUFFMAN, G4_CODEC_LSOP08, G4_CODEC_LSOP12, G4_DECLINED,
                   G4_ELEM_F32, G4_ELEM_I16, G4_ELEM_I32, G4_ELEM_ICF, G4_LSOP12_NO_DEFLATE, G4_LSOP12_VALUE_CHECKSUM, G4_MEM_DEVICE,
                   G4_MEM_HOST, G4_OK, BandDesc, CodecList, IcfDesc, check)

from .stats import AnalysisMixin  # noqa: E402

INT4_NULL_CODE = -(2 ** 31)  # util/GridfourConstants.java:61


class Context:
    """One CUDA stream + scratch (g4_context).  Not shareable between threads: Context.default() hands every THREAD its
    own context per device (the reference enters one decoder instance from the application thread and from the
    read-ahead thread, TileDecompressionAssistant.java:88; here each of them works on its own stream and scratch)."""

    _default = threading.local()

    def __init__(self, device=0, stream=None):
        self._h = C.c_void_p()
        check(_lib.lib().g4_context_create(int(device), C.c_void_p(stream) if stream else None, C.byref(self._h)),
              "g4_context_create")
        self.device = device

    @classmethod
    def default(cls, device=0):
        table = getattr(cls._default, "table", None)
        if table is None:
            table = cls._default.table = {}
        if device not in table:
            table[device] = cls(device)
        return table[device]

    def after_torch_stream(self, device):
        """Device tensors produced by kernels still pending on torch's current stream are complete before this context's
        next launch (g4_context_order_stream, events only)."""
        import torch

        check(_lib.lib().g4_context_order_stream(self._h, C.c_void_p(torch.cuda.current_stream(device).cuda_stream), 1),
              "g4_context_order_stream")

    def before_torch_stream(self, device):
        """torch's current stream continues only after everything this context has launched so far."""
        import torch

        check(_lib.lib().g4_context_order_stream(self._h, C.c_void_p(torch.cuda.current_stream(device).cuda_stream), 0),
              "g4_context_order_stream")

    def synchronize(self):
        check(_lib.lib().g4_context_synchronize(self._h))

    @property
    def launch_count(self):
        return int(_lib.lib().g4_launch_count(self._h))

    def set_async(self, enabled):
        """Device batches are only enqueued on the context's stream (decodeTiles returns at once, the per-tile status tensor
        is valid after synchronize()): lets a caller keep several windows of tiles in flight."""
        check(_lib.lib().g4_context_set_async(self._h, int(bool(enabled))))

    def set_timing(self, enabled):
        check(_lib.lib().g4_context_set_timing(self._h, int(bool(enabled))))

    def kernel_time_ms(self, direction, codec_kind):
        """Device time of the latest decode (0) / encode (1) kernel launch of a codec kind; None if not run."""
        ms = _lib.lib().g4_kernel_time_ms(self._h, direction, codec_kind)
        return None if ms < 0 else ms

    def fill_terrain(self, device_ptr, elem_type, row0, col0, n_rows, n_cols, seed=0x9E3779B97F4A7C15):
        check(_lib.lib().g4_fill_terrain(self._h, elem_type, C.c_uint64(seed), row0, col0, n_rows, n_cols,
                                         C.c_void_p(device_ptr)), "g4_fill_terrain")

    def close(self):
        if self._h:
            _lib.lib().g4_context_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ICompressionEncoder:
    """compress/ICompressionEncoder.java:46-92"""

    codec_id = None

    def __init__(self, context=None):
        self._ctx = context

    def _context(self):
        return self._ctx or Context.default()

    def native_id(self):
        """The codec id this instance passes to the library, with its option bits (include/g4codec.h)."""
        return self.codec_id

    def implementsIntegerEncoding(self):
        return self.codec_id != G4_CODEC_FLOAT

    def implementsFloatingPointEncoding(self):
        return self.codec_id == G4_CODEC_FLOAT

    def encode(self, codecIndex, nRows, nCols, values):
        """Returns the packing bytes, or None where the Java codec returns null."""
        if not self.implementsIntegerEncoding():
            raise ValueError("codec does not implement integer encoding")  # CodecFloat.java:116-125
        v = np.ascontiguousarray(values, dtype=np.int32).reshape(-1)
        if v.size != nRows * nCols:
            raise ValueError("values.length != nRows*nCols")
        cap = v.size * 6 + 1024
        out = np.empty(cap, np.uint8)
        n = C.c_size_t(0)
        pred = C.c_int(0)
        st = _lib.lib().g4_encode_i32(self._context()._h, self.native_id(), int(codecIndex), int(nRows), int(nCols), v.ctypes.data,
                                      out.ctypes.data, cap, C.byref(n), C.byref(pred))
        if st == G4_DECLINED:
            return None
        check(st, "g4_encode_i32")
        self.lastPredictor = pred.value
        return out[: n.value].tobytes()

    def encodeFloats(self, codecIndex, nRows, nCols, values):
        if not self.implementsFloatingPointEncoding():
            return None  # CodecHuffman.java:241-244
        v = np.ascontiguousarray(values, dtype=np.float32).reshape(-1)
        if v.size != nRows * nCols:
            raise ValueError("values.length != nRows*nCols")
        cap = v.size * 6 + 4096
        out = np.empty(cap, np.uint8)
        n = C.c_size_t(0)
        st = _lib.lib().g4_encode_f32(self._context()._h, self.codec_id, int(codecIndex), int(nRows), int(nCols), v.ctypes.data,
                                      out.ctypes.data, cap, C.byref(n))
        if st == G4_DECLINED:
            return None
        check(st, "g4_encode_f32")
        return out[: n.value].tobytes()


class ICompressionDecoder:
    """compress/ICompressionDecoder.java:49-107"""

    codec_id = None

    def __init__(self, context=None):
        self._ctx = context

    def _context(self):
        return self._ctx or Context.default()

    def decode(self, nRows, nColumns, packing):
        """Returns int32[nRows, nColumns]; raises FormatError (an IOError) on malformed input."""
        if self.codec_id == G4_CODEC_FLOAT:
            raise ValueError("codec does not implement integer decoding")
        b = np.frombuffer(bytes(packing), dtype=np.uint8)
        out = np.empty((nRows, nColumns), np.int32)
        st = _lib.lib().g4_decode_i32(self._context()._h, self.codec_id, int(nRows), int(nColumns), b.ctypes.data, b.size,
                                      out.ctypes.data)
        if st == G4_DECLINED:
            return None
        check(st, "g4_decode_i32")
        return out

    def decodeFloats(self, nRows, nColumns, packing):
        if self.codec_id != G4_CODEC_FLOAT:
            return None
        b = np.frombuffer(bytes(packing), dtype=np.uint8)
        out = np.empty((nRows, nColumns), np.float32)
        st = _lib.lib().g4_decode_f32(self._context()._h, self.codec_id, int(nRows), int(nColumns), b.ctypes.data, b.size,
                                      out.ctypes.data)
        if st == G4_DECLINED:
            return None
        check(st, "g4_decode_f32")
        return out

    # analysis hooks of the interface: the M32-based codecs (CodecHuffman, CodecDeflate) implement them through
    # g4_analyze_tiles (stats.AnalysisMixin); the others keep no statistics here
    def analyze(self, nRows, nColumns, packing):
        pass

    def reportAnalysisData(self, ps, nTilesInRaster):
        pass

    def clearAnalysisData(self):
        pass


class _Codec(ICompressionEncoder, ICompressionDecoder):
    def __init__(self, context=None):
        ICompressionEncoder.__init__(self, context)


class CodecHuffman(AnalysisMixin, _Codec):
    """compress/CodecHuffman.java"""
    codec_id = G4_CODEC_HUFFMAN
    _report_title = "Gridfour_Huffman"
    _with_tree = True


class CodecDeflate(AnalysisMixin, _Codec):
    """compress/CodecDeflate.java"""
    codec_id = G4_CODEC_DEFLATE
    _report_title = "Gridfour_Deflate"


class CodecFloat(_Codec):
    """compress/CodecFloat.java"""
    codec_id = G4_CODEC_FLOAT


class CodecCanonHuffman(_Codec):
    """compress/canonicalHuffman/CodecCanonHuffman.java"""
    codec_id = G4_CODEC_CANON_HUFFMAN


class LsEncoder12(ICompressionEncoder):
    """lsop/LsEncoder12.java, with its two switches (:93-119): the Deflate alternative (on by default) and the value
    checksum (off by default)."""
    codec_id = G4_CODEC_LSOP12

    def __init__(self, context=None):
        super().__init__(context)
        self.deflateEnabled = True
        self.valueChecksumEnabled = False

    def setDeflateEnabled(self, deflateEnabled):
        """False: every packing is the canonical-Huffman form; the Deflate alternative is not tried."""
        self.deflateEnabled = bool(deflateEnabled)

    def isDeflateEnabled(self):
        return self.deflateEnabled

    def setValueChecksumEnabled(self, valueChecksumEnabled):
        """True: every packing carries the CRC-32C of the tile's values, which the decoder checks."""
        self.valueChecksumEnabled = bool(valueChecksumEnabled)

    def isValueChecksumEnabled(self):
        return self.valueChecksumEnabled

    def native_id(self):
        return self.codec_id | (0 if self.deflateEnabled else G4_LSOP12_NO_DEFLATE) | (
            G4_LSOP12_VALUE_CHECKSUM if self.valueChecksumEnabled else 0)


class LsDecoder12(ICompressionDecoder):
    """lsop/LsDecoder12.java"""
    codec_id = G4_CODEC_LSOP12


class LsDecoder08(ICompressionDecoder):
    """lsop/LsDecoder08.java -- the legacy 8-coefficient codec, decode only (the reference no longer registers it,
    lsop/LsCodecUtility.java:73)."""
    codec_id = G4_CODEC_LSOP08


class LsEncoder08(ICompressionEncoder):
    """lsop/LsEncoder08.java is not built on the GPU: every encode is declined (None), so CodecMaster falls through to the
    next codec or to raw storage.  The class exists so that a codec list naming LSOP08 can be registered for reading."""
    codec_id = G4_CODEC_LSOP08


_STANDARD = {
    "GvrsHuffman": (CodecHuffman, CodecHuffman),
    "GvrsDeflate": (CodecDeflate, CodecDeflate),
    "GvrsFloat": (CodecFloat, CodecFloat),
    "GvrsCanonicalHuffman": (CodecCanonHuffman, CodecCanonHuffman),
    "LSOP12": (LsEncoder12, LsDecoder12),
    "LSOP08": (LsEncoder08, LsDecoder08),
}


class CodecSpecification:
    """The codec-list part of GvrsFileSpecification (gvrs/GvrsFileSpecification.java:221-230,1535-1724).

    Position in the list is the codec index stored in packing[0].  The default list mirrors the reference's:
    GvrsHuffman, GvrsDeflate, GvrsFloat (the 1.0.6 snapshot's decode-only legacy Huffman entry is kept as a
    full codec here because BASELINE.json names CodecHuffman encode explicitly; SURVEY.md note N1).
    """

    def __init__(self, default=True):
        self.codecList = []  # [(id, encoderClass, decoderClass)]
        if default:
            for cid in ("GvrsHuffman", "GvrsDeflate", "GvrsFloat"):
                self.addCompressionCodec(cid, *_STANDARD[cid])

    def addCompressionCodec(self, codecID, encoder, decoder=None):
        """addCompressionCodec(id, codecClass) or (id, encoderClass, decoderClass); same id replaces and moves to
        the end of the list (GvrsFileSpecification.java:1590,1628-1630)."""
        decoder = decoder or encoder
        if not codecID or len(codecID) > 32 or not codecID.replace("_", "a").isalnum() or codecID[0].isdigit():
            raise ValueError("invalid codec identification: %r" % (codecID,))
        if not issubclass(encoder, ICompressionEncoder) or not issubclass(decoder, ICompressionDecoder):
            raise ValueError("codec classes must implement ICompressionEncoder / ICompressionDecoder")
        self.codecList = [c for c in self.codecList if c[0] != codecID]
        if len(self.codecList) >= 255:
            raise ValueError("maximum number of compression codecs is 255")
        self.codecList.append((codecID, encoder, decoder))

    def removeAllCompressionCodecs(self):
        self.codecList = []

    def removeCompressionCodec(self, codecID):
        n = len(self.codecList)
        self.codecList = [c for c in self.codecList if c[0] != codecID]
        return len(self.codecList) != n

    def getCompressionCodecs(self):
        return list(self.codecList)

    def native_list(self):
        cl = CodecList()
        cl.n_codecs = len(self.codecList)
        for k, (cid, enc, _dec) in enumerate(self.codecList):
            cl.codec_ids[k] = enc.codec_id
        return cl


class IntCodedFloat:
    """The mapping of an integer-coded float element (GvrsElementIntCodedFloat): float values are stored as int codes,
    code = floor((v - offset) * scale + 0.5), and read back as code / scale + offset; NaN <-> fill_int <-> fill_value.
    The exact arithmetic is that of g4_icf_desc (include/g4codec.h).  The maps run on the GPU (g4_icf_map)."""

    def __init__(self, scale, offset=0.0, fill_int=INT4_NULL_CODE, fill_value=float("nan")):
        self.scale, self.offset, self.fill_value = np.float32(scale), np.float32(offset), np.float32(fill_value)
        self.fill_int = int(fill_int)
        if not np.isfinite(self.scale) or self.scale == 0:
            raise ValueError("integer-coded float: the scale must be finite and not zero")

    def desc(self):
        d = IcfDesc()
        d.scale, d.offset, d.fill_int, d.fill_value = float(self.scale), float(self.offset), self.fill_int, float(self.fill_value)
        return d

    def __eq__(self, other):
        return isinstance(other, IntCodedFloat) and (self.scale, self.offset, self.fill_int) == (other.scale, other.offset, other.fill_int) \
            and self.fill_value.tobytes() == other.fill_value.tobytes()

    def __repr__(self):
        return "IntCodedFloat(scale=%r, offset=%r, fill_int=%d, fill_value=%r)" % (float(self.scale), float(self.offset), self.fill_int,
                                                                                  float(self.fill_value))

    def to_float(self, codes, out=None, context=None):
        """int32 codes -> float32 values (numpy, or a torch CUDA tensor); `out` may be `codes` viewed as float32."""
        return self._map(1, codes, out, np.int32, np.float32, context)

    def to_int(self, values, out=None, context=None):
        """float32 values -> int32 codes (numpy, or a torch CUDA tensor)."""
        return self._map(0, values, out, np.float32, np.int32, context)

    def _map(self, to_float, src, out, src_dt, dst_dt, context):
        ctx = context or Context.default()
        d = self.desc()
        if isinstance(src, np.ndarray):
            src = np.asarray(src, dtype=src_dt)
            if src.ndim == 1:
                src = src.reshape(1, -1)
            out = np.empty(src.shape, dst_dt) if out is None else out
            if out.dtype != dst_dt or out.shape != src.shape:
                raise ValueError("out: %s of shape %s" % (np.dtype(dst_dt).name, src.shape))
            sp, dp = _pitch(src.strides, src.itemsize), _pitch(out.strides, out.itemsize)
            if src.size:
                check(_lib.lib().g4_icf_map(ctx._h, to_float, C.byref(d), G4_MEM_HOST, src.shape[0], src.shape[1], src.ctypes.data, sp,
                                            out.ctypes.data, dp), "g4_icf_map")
            return out
        import torch

        tdt = {np.int32: torch.int32, np.float32: torch.float32}
        if not (isinstance(src, torch.Tensor) and src.is_cuda and src.dtype == tdt[src_dt] and src.dim() == 2):
            raise ValueError("a 2-D %s numpy array or CUDA tensor" % np.dtype(src_dt).name)
        out = torch.empty(src.shape, dtype=tdt[dst_dt], device=src.device) if out is None else out
        if out.dtype != tdt[dst_dt] or tuple(out.shape) != tuple(src.shape):
            raise ValueError("out: %s of shape %s" % (np.dtype(dst_dt).name, tuple(src.shape)))
        sp, dp = _pitch(tuple(4 * x for x in src.stride()), 4), _pitch(tuple(4 * x for x in out.stride()), 4)
        if src.numel():
            ctx.after_torch_stream(src.device)
            st = _lib.lib().g4_icf_map(ctx._h, to_float, C.byref(d), G4_MEM_DEVICE, src.shape[0], src.shape[1], src.data_ptr(), sp,
                                       out.data_ptr(), dp)
            ctx.before_torch_stream(src.device)
            check(st, "g4_icf_map")
        return out


def _pitch(strides, itemsize):
    """Samples per row of a 2-D array whose rows are contiguous."""
    if strides[1] != itemsize or strides[0] % itemsize or strides[0] < 0:
        raise ValueError("rows must be contiguous, with a non-negative pitch that is a whole number of samples")
    return strides[0] // itemsize


class TileBatch:
    """Result of CodecMaster.encodeTiles: payloads packed back to back (8-byte aligned) in `arena`.  `icf` is the
    IntCodedFloat of a batch of integer-coded float tiles (its payloads hold the codes; decodeTiles returns float32)."""

    def __init__(self, arena, offsets, lens, codec, predictor, status, total_bytes, band, icf=None):
        self.arena, self.offsets, self.lens = arena, offsets, lens
        self.codec, self.predictor, self.status = codec, predictor, status
        self.total_bytes, self.band, self.icf = total_bytes, band, icf

    def payload(self, t):
        o, n = int(self.offsets[t]), int(self.lens[t])
        return bytes(np.asarray(self.arena[o:o + n]).tobytes())


class CodecMaster:
    """gvrs/CodecMaster.java:142-203 + the new batched entry points."""

    def __init__(self, spec=None, context=None):
        self.spec = spec or CodecSpecification()
        self._ctx = context
        self._enc = [enc(context) for (_i, enc, _d) in self.spec.codecList]
        self._dec = [dec(context) for (_i, _e, dec) in self.spec.codecList]

    def _context(self):
        return self._ctx or Context.default()

    def getEncoder(self, codecID):
        """The encoder instance this master encodes with for the codec named codecID (e.g. "LSOP12"), so that its options
        can be set; None when the list has no such codec."""
        for (cid, _e, _d), enc in zip(self.spec.codecList, self._enc):
            if cid == codecID:
                return enc
        return None

    def _native_list(self):
        """The codec list of the native calls, taken from this master's encoder instances (with their option bits)."""
        cl = CodecList()
        cl.n_codecs = len(self._enc)
        for k, enc in enumerate(self._enc):
            cl.codec_ids[k] = enc.native_id()
        return cl

    # -- per tile, exactly CodecMaster.encodeSingleThread / decode ---------------------------------------
    def encode(self, nRows, nCols, values):
        result = None
        for k, codec in enumerate(self._enc):
            if codec.implementsIntegerEncoding():
                test = codec.encode(k, nRows, nCols, values)
                if test is not None and (result is None or len(test) < len(result)):
                    result = test
        return result

    def encodeFloats(self, nRows, nCols, values):
        result = None
        for k, codec in enumerate(self._enc):
            if codec.implementsFloatingPointEncoding():
                test = codec.encodeFloats(k, nRows, nCols, values)
                if test is not None and (result is None or len(test) < len(result)):
                    result = test
        return result

    def decode(self, nRows, nColumns, packing):
        index = packing[0] & 0xFF
        if index >= len(self._dec):
            raise IOError("Invalid compression-type code %d" % index)  # CodecMaster.java:197-199
        return self._dec[index].decode(nRows, nColumns, packing)

    def decodeFloats(self, nRows, nColumns, packing):
        index = packing[0] & 0xFF
        if index >= len(self._dec):
            raise IOError("Invalid compression-type code %d" % index)
        return self._dec[index].decodeFloats(nRows, nColumns, packing)

    # -- batched (new): a band of tiles in one call -------------------------------------------------------
    @staticmethod
    def _band(grid_shape, dtype, tileRows, tileCols, pitch=None, fillValue=None):
        rows, cols = grid_shape
        if rows % tileRows or cols % tileCols:
            raise ValueError("grid dimensions must be multiples of the tile size (GVRS tiles are full size)")
        b = BandDesc()
        dt = np.dtype(dtype)
        b.elem_type = G4_ELEM_F32 if dt == np.float32 else G4_ELEM_I16 if dt == np.int16 else G4_ELEM_I32
        # TileElementShort: the element's fill value is coded as null (gvrs/TileElementShort.java:213-218); the default
        # fill of a short element is SHORT_NULL_CODE
        b.fill_value = int(fillValue) if fillValue is not None else -32768
        b.tile_rows, b.tile_cols = tileRows, tileCols
        b.tiles_down, b.tiles_across = rows // tileRows, cols // tileCols
        b.grid_pitch = pitch or cols
        return b

    def _encode_call(self, icf):
        """g4_encode_tiles, or g4_encode_tiles_icf with the descriptor of `icf` bound in."""
        L = _lib.lib()
        if icf is None:
            return L.g4_encode_tiles, "g4_encode_tiles"
        d = icf.desc()
        return (lambda ctx, cl, band, *rest: L.g4_encode_tiles_icf(ctx, cl, band, C.byref(d), *rest)), "g4_encode_tiles_icf"

    def encodeTiles(self, grid, tileRows, tileCols, fillValue=None, icf=None, padValue=None):
        """grid: 2-D numpy array (host path) or torch CUDA tensor (device path); int32, float32, or int16 (a short
        element, TileElementShort: `fillValue` is coded as null, raw tiles take 2 bytes per sample).  With `icf` (an
        IntCodedFloat) the float32 grid is an integer-coded float element: it is mapped to codes on the GPU and the codes are
        encoded with the integer codecs; the batch remembers the mapping.
        With `padValue` (CUDA tensors only) the grid may have any dimensions and any row pitch, as long as its rows are
        contiguous: it covers ceil(rows / tileRows) x ceil(cols / tileCols) tiles, whose cells outside the grid encode as
        padValue does (g4_encode_window; the padding happens on the device)."""
        if padValue is not None:
            if isinstance(grid, np.ndarray):
                raise ValueError("padValue: CUDA tensors only (a numpy grid is padded by the caller)")
            return self._encode_window(grid, tileRows, tileCols, fillValue, icf, padValue)
        L = _lib.lib()
        cl = self._native_list()
        total = C.c_uint64(0)
        encode, name = self._encode_call(icf)
        if isinstance(grid, np.ndarray):
            g = np.ascontiguousarray(grid)
            if g.dtype not in (np.int32, np.float32, np.int16) or (icf is not None and g.dtype != np.float32):
                raise ValueError("int32, float32 or int16 rasters only (float32 for an integer-coded float element)")
            band = self._band(g.shape, g.dtype, tileRows, tileCols, fillValue=fillValue)
            if icf is not None:
                band.elem_type = G4_ELEM_ICF
            nT = band.tiles_down * band.tiles_across
            cap = int(L.g4_encode_arena_bound(C.byref(band)))
            arena = np.empty(cap, np.uint8)
            offsets = np.empty(nT, np.uint64)
            lens = np.empty(nT, np.uint32)
            codec = np.empty(nT, np.uint8)
            pred = np.empty(nT, np.uint8)
            status = np.empty(nT, np.int32)
            st = encode(self._context()._h, C.byref(cl), C.byref(band), G4_MEM_HOST, g.ctypes.data, arena.ctypes.data, cap,
                        offsets.ctypes.data, lens.ctypes.data, codec.ctypes.data, pred.ctypes.data, status.ctypes.data, C.byref(total))
            check(st, name)
            return TileBatch(arena[: total.value], offsets, lens, codec, pred, status, total.value, band, icf)
        import torch

        if not (isinstance(grid, torch.Tensor) and grid.is_cuda and grid.dim() == 2 and grid.is_contiguous()):
            raise ValueError("expected a contiguous 2-D CUDA tensor")
        if icf is not None and grid.dtype != torch.float32:
            raise ValueError("an integer-coded float element is encoded from a float32 tensor")
        npdt = np.float32 if grid.dtype == torch.float32 else np.int16 if grid.dtype == torch.int16 else np.int32
        band = self._band(tuple(grid.shape), npdt, tileRows, tileCols, fillValue=fillValue)
        if icf is not None:
            band.elem_type = G4_ELEM_ICF
        nT = band.tiles_down * band.tiles_across
        cap = int(L.g4_encode_arena_bound(C.byref(band)))
        dev = grid.device
        arena = torch.empty(cap, dtype=torch.uint8, device=dev)
        offsets = torch.empty(nT, dtype=torch.int64, device=dev)
        lens = torch.empty(nT, dtype=torch.int32, device=dev)
        codec = torch.empty(nT, dtype=torch.uint8, device=dev)
        pred = torch.empty(nT, dtype=torch.uint8, device=dev)
        status = torch.empty(nT, dtype=torch.int32, device=dev)
        ctx = self._context()
        ctx.after_torch_stream(dev)  # `grid` may come from kernels still queued on torch's stream
        st = encode(ctx._h, C.byref(cl), C.byref(band), G4_MEM_DEVICE, grid.data_ptr(), arena.data_ptr(), cap, offsets.data_ptr(),
                    lens.data_ptr(), codec.data_ptr(), pred.data_ptr(), status.data_ptr(), C.byref(total))
        ctx.before_torch_stream(dev)
        check(st, name)
        return TileBatch(arena, offsets, lens, codec, pred, status, total.value, band, icf)

    def _encode_window(self, grid, tileRows, tileCols, fillValue, icf, padValue):
        """encodeTiles of a CUDA tensor of any dimensions, padded with padValue on the device (g4_encode_window)."""
        import torch

        L = _lib.lib()
        dtypes = {torch.int32: np.int32, torch.float32: np.float32, torch.int16: np.int16}
        if not (isinstance(grid, torch.Tensor) and grid.is_cuda and grid.dim() == 2 and grid.dtype in dtypes):
            raise ValueError("expected a 2-D int32, float32 or int16 CUDA tensor")
        if icf is not None and grid.dtype != torch.float32:
            raise ValueError("an integer-coded float element is encoded from a float32 tensor")
        rows, cols = grid.shape
        if rows < 1 or cols < 1:
            raise ValueError("an empty grid")
        if (cols > 1 and grid.stride(1) != 1) or (rows > 1 and grid.stride(0) < cols):
            raise ValueError("the grid's rows must be contiguous")
        pitch = grid.stride(0) if rows > 1 else cols
        npdt = dtypes[grid.dtype]
        b = BandDesc()
        b.elem_type = G4_ELEM_F32 if npdt == np.float32 else G4_ELEM_I16 if npdt == np.int16 else G4_ELEM_I32
        if icf is not None:
            b.elem_type = G4_ELEM_ICF
        b.fill_value = int(fillValue) if fillValue is not None else -32768
        b.tile_rows, b.tile_cols = tileRows, tileCols
        b.tiles_down, b.tiles_across = -(-rows // tileRows), -(-cols // tileCols)
        b.grid_pitch = b.tiles_across * tileCols
        # the margin sample as a 32-bit pattern of the source type (int16: the low half)
        fill_bits = int(np.array(padValue, dtype=npdt).view(np.uint16 if npdt == np.int16 else np.uint32))
        nT = b.tiles_down * b.tiles_across
        cap = int(L.g4_encode_arena_bound(C.byref(b)))
        dev = grid.device
        arena = torch.empty(cap, dtype=torch.uint8, device=dev)
        offsets = torch.empty(nT, dtype=torch.int64, device=dev)
        lens = torch.empty(nT, dtype=torch.int32, device=dev)
        codec = torch.empty(nT, dtype=torch.uint8, device=dev)
        pred = torch.empty(nT, dtype=torch.uint8, device=dev)
        status = torch.empty(nT, dtype=torch.int32, device=dev)
        d = icf.desc() if icf is not None else None
        total = C.c_uint64(0)
        ctx = self._context()
        ctx.after_torch_stream(dev)  # `grid` may come from kernels still queued on torch's stream
        st = L.g4_encode_window(ctx._h, C.byref(self._native_list()), C.byref(b), None if d is None else C.byref(d), rows, cols,
                                grid.data_ptr(), pitch, fill_bits, arena.data_ptr(), cap, offsets.data_ptr(), lens.data_ptr(),
                                codec.data_ptr(), pred.data_ptr(), status.data_ptr(), C.byref(total))
        ctx.before_torch_stream(dev)
        check(st, "g4_encode_window")
        return TileBatch(arena, offsets, lens, codec, pred, status, total.value, b, icf)

    # -- tile lists (new): scattered tiles of one size, each with its own {offset, pitch} -- the tile cache's calls -----
    @staticmethod
    def _refs(refs):
        from ._lib import TileRef

        arr = (TileRef * len(refs))()
        for k, (off, pitch) in enumerate(refs):
            arr[k].offset, arr[k].pitch = int(off), int(pitch)
        return arr

    def encodeTileList(self, base, refs, tileRows, tileCols):
        """base: numpy array (host) or torch CUDA tensor holding the tiles; refs: [(offset, pitch)] in samples from base's
        first element (RasterTileCache.flush: whatever tiles are dirty, gvrs/RasterTileCache.java:286-294).  Returns a
        TileBatch whose tile t is list position t."""
        L = _lib.lib()
        cl = self._native_list()
        n = len(refs)
        total = C.c_uint64(0)
        tiles = self._refs(refs)
        cap = n * 4 * tileRows * tileCols + 64
        if isinstance(base, np.ndarray):
            if base.dtype not in (np.int32, np.float32) or not base.flags["C_CONTIGUOUS"]:
                raise ValueError("a contiguous int32 or float32 array")
            elem = G4_ELEM_F32 if base.dtype == np.float32 else G4_ELEM_I32
            arena, offsets, lens = np.empty(cap, np.uint8), np.empty(n, np.uint64), np.empty(n, np.uint32)
            codec, pred, status = np.empty(n, np.uint8), np.empty(n, np.uint8), np.empty(n, np.int32)
            st = L.g4_encode_tile_list(self._context()._h, C.byref(cl), elem, tileRows, tileCols, n, G4_MEM_HOST, base.ctypes.data, tiles,
                                       arena.ctypes.data, cap, offsets.ctypes.data, lens.ctypes.data, codec.ctypes.data, pred.ctypes.data,
                                       status.ctypes.data, C.byref(total))
            check(st, "g4_encode_tile_list")
            band = self._band((tileRows, n * tileCols), base.dtype, tileRows, tileCols)
            return TileBatch(arena[: total.value], offsets, lens, codec, pred, status, total.value, band)
        import torch

        if not (isinstance(base, torch.Tensor) and base.is_cuda and base.is_contiguous()):
            raise ValueError("expected a contiguous CUDA tensor")
        elem = G4_ELEM_F32 if base.dtype == torch.float32 else G4_ELEM_I32
        dev = base.device
        arena = torch.empty(cap, dtype=torch.uint8, device=dev)
        offsets = torch.empty(n, dtype=torch.int64, device=dev)
        lens = torch.empty(n, dtype=torch.int32, device=dev)
        codec, pred = torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)
        status = torch.empty(n, dtype=torch.int32, device=dev)
        ctx = self._context()
        ctx.after_torch_stream(dev)
        st = L.g4_encode_tile_list(ctx._h, C.byref(cl), elem, tileRows, tileCols, n, G4_MEM_DEVICE, base.data_ptr(), tiles, arena.data_ptr(), cap,
                                   offsets.data_ptr(), lens.data_ptr(), codec.data_ptr(), pred.data_ptr(), status.data_ptr(), C.byref(total))
        ctx.before_torch_stream(dev)
        check(st, "g4_encode_tile_list")
        band = self._band((tileRows, n * tileCols), np.float32 if elem == G4_ELEM_F32 else np.int32, tileRows, tileCols)
        return TileBatch(arena, offsets, lens, codec, pred, status, total.value, band)

    def decodeTileList(self, arena, offsets, lens, base, refs, tileRows, tileCols):
        """Decodes payload t (arena[offsets[t] : +lens[t]]) into the tile at refs[t] of `base` (numpy or torch CUDA; all
        buffers in the same memory space).  RasterTileCache.readTileUsingAssistant / a bulk readBlock
        (gvrs/RasterTileCache.java:339-426, gvrs/GvrsElement.java:298-404): every missing tile of a window in one call."""
        L = _lib.lib()
        cl = self._native_list()
        n = len(refs)
        tiles = self._refs(refs)
        if isinstance(base, np.ndarray):
            if base.dtype not in (np.int32, np.float32) or not base.flags["C_CONTIGUOUS"]:
                raise ValueError("a contiguous int32 or float32 array")
            elem = G4_ELEM_F32 if base.dtype == np.float32 else G4_ELEM_I32
            a = np.frombuffer(arena, dtype=np.uint8) if not isinstance(arena, np.ndarray) else np.ascontiguousarray(arena)
            off = np.ascontiguousarray(offsets, dtype=np.uint64)
            ln = np.ascontiguousarray(lens, dtype=np.uint32)
            status = np.empty(n, np.int32)
            st = L.g4_decode_tile_list(self._context()._h, C.byref(cl), elem, tileRows, tileCols, n, G4_MEM_HOST, a.ctypes.data, int(a.size),
                                       off.ctypes.data, ln.ctypes.data, base.ctypes.data, tiles, status.ctypes.data)
            self.lastStatus = status
            check(st, "g4_decode_tile_list")
            return base
        import torch

        elem = G4_ELEM_F32 if base.dtype == torch.float32 else G4_ELEM_I32
        status = torch.empty(n, dtype=torch.int32, device=base.device)
        ctx = self._context()
        ctx.after_torch_stream(base.device)
        st = L.g4_decode_tile_list(ctx._h, C.byref(cl), elem, tileRows, tileCols, n, G4_MEM_DEVICE, arena.data_ptr(), int(arena.numel()),
                                   offsets.data_ptr(), lens.data_ptr(), base.data_ptr(), tiles, status.data_ptr())
        ctx.before_torch_stream(base.device)
        self.lastStatus = status
        check(st, "g4_decode_tile_list")
        return base

    def decodeImageTiles(self, image, payload_offsets, lens, status, tilesDown, tilesAcross, tileRows, tileCols, dtype, fillValue,
                         icf=None):
        """Decodes the tiles of a one-element raster whose payloads sit inside a GVRS file image (gvrs.GvrsImage.read_raster):
        the image is the arena of g4_decode_tiles.  Tiles the file does not hold (status G4_DECLINED) are pointed at one
        raw tile of fill values appended to the arena (RasterTile.setToNullState).  With `icf` (an IntCodedFloat; dtype
        int32, fillValue its fill_int) the codes are mapped and the raster comes back as float32."""
        from ._lib import G4_DECLINED

        band = self._band((tilesDown * tileRows, tilesAcross * tileCols), dtype, tileRows, tileCols,
                          fillValue=fillValue if np.dtype(dtype) == np.int16 else None)
        if icf is not None:
            band.elem_type = G4_ELEM_ICF
        arena = np.frombuffer(image, dtype=np.uint8) if not isinstance(image, np.ndarray) else image
        offsets = np.array(payload_offsets, dtype=np.uint64)
        lens = np.array(lens, dtype=np.uint32)
        absent = np.asarray(status) == G4_DECLINED
        if absent.any():
            fill = np.full(tileRows * tileCols, fillValue, dtype=np.dtype(dtype)).tobytes()
            fill += bytes((-len(fill)) & 3)
            base = (arena.size + 7) & ~7
            arena = np.concatenate([arena, np.zeros(base - arena.size, np.uint8), np.frombuffer(fill, dtype=np.uint8)])
            offsets[absent] = base
            lens[absent] = len(fill)
        return self.decodeTiles(TileBatch(arena, offsets, lens, None, None, None, int(arena.size), band, icf))

    def _decode_call(self, icf):
        """g4_decode_tiles_bounded, or g4_decode_tiles_icf with the descriptor of `icf` bound in."""
        L = _lib.lib()
        if icf is None:
            return L.g4_decode_tiles_bounded, "g4_decode_tiles"
        d = icf.desc()
        return (lambda ctx, cl, band, *rest: L.g4_decode_tiles_icf(ctx, cl, band, C.byref(d), *rest)), "g4_decode_tiles_icf"

    def decodeTiles(self, batch, out=None):
        """Inverse of encodeTiles.  Returns the raster (numpy for host batches, torch for device batches); float32 for a
        batch of integer-coded float tiles (batch.icf)."""
        cl = self._native_list()
        band = batch.band
        rows, cols = band.tiles_down * band.tile_rows, band.tiles_across * band.tile_cols
        decode, name = self._decode_call(batch.icf)
        f32 = band.elem_type in (G4_ELEM_F32, G4_ELEM_ICF)
        if isinstance(batch.arena, np.ndarray):
            dt = np.float32 if f32 else np.int16 if band.elem_type == G4_ELEM_I16 else np.int32
            grid = out if out is not None else np.empty((rows, cols), dt)
            status = np.empty(band.tiles_down * band.tiles_across, np.int32)
            arena = np.ascontiguousarray(batch.arena)
            offsets = np.ascontiguousarray(batch.offsets, dtype=np.uint64)
            lens = np.ascontiguousarray(batch.lens, dtype=np.uint32)
            st = decode(self._context()._h, C.byref(cl), C.byref(band), G4_MEM_HOST, arena.ctypes.data, int(arena.size), offsets.ctypes.data,
                        lens.ctypes.data, grid.ctypes.data, status.ctypes.data)
            self.lastStatus = status
            check(st, name)
            return grid
        import torch

        dt = torch.float32 if f32 else torch.int16 if band.elem_type == G4_ELEM_I16 else torch.int32
        grid = out if out is not None else torch.empty((rows, cols), dtype=dt, device=batch.arena.device)
        status = torch.empty(band.tiles_down * band.tiles_across, dtype=torch.int32, device=batch.arena.device)
        ctx = self._context()
        ctx.after_torch_stream(batch.arena.device)  # the payloads and `out` may still be in use on torch's stream
        st = decode(ctx._h, C.byref(cl), C.byref(band), G4_MEM_DEVICE, batch.arena.data_ptr(), int(batch.arena.numel()),
                    batch.offsets.data_ptr(), batch.lens.data_ptr(), grid.data_ptr(), status.data_ptr())
        ctx.before_torch_stream(batch.arena.device)
        self.lastStatus = status
        check(st, name)
        return grid
