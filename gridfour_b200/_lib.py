"""ctypes binding of libg4codec.so (the C ABI of include/g4codec.h).

The CUDA library is the only compute path: importing this module fails loudly when the shared object has
not been built (run `python -c "import __graft_entry__ as g; g.build()"` or `make -C gridfour_b200/csrc`).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libg4codec.so")

G4_OK, G4_DECLINED, G4_CHECKSUM_MISMATCH = 0, 1, 2
G4_ERR_ARG, G4_ERR_FORMAT, G4_ERR_CAPACITY, G4_ERR_CUDA, G4_ERR_UNSUPPORTED = -1, -2, -3, -4, -5
G4_CODEC_HUFFMAN, G4_CODEC_DEFLATE, G4_CODEC_FLOAT, G4_CODEC_CANON_HUFFMAN, G4_CODEC_LSOP12 = 0, 1, 2, 3, 4
G4_CODEC_LSOP08 = 5
G4_LSOP12_NO_DEFLATE, G4_LSOP12_VALUE_CHECKSUM = 1 << 8, 1 << 9  # option bits of an LSOP12 codec entry
G4_ELEM_I32, G4_ELEM_F32, G4_ELEM_I16, G4_ELEM_ICF = 0, 1, 2, 3
G4_MEM_HOST, G4_MEM_DEVICE = 0, 1
G4_MAX_CODECS = 16
G4_CODEC_RAW = 255

# every symbol include/g4codec.h declares (checked by tests/test_abi.py)
EXPORTS = [
    "g4_abi_version", "g4_status_string", "g4_last_error", "g4_device_count", "g4_codec_id_from_name", "g4_codec_name",
    "g4_context_create", "g4_context_destroy", "g4_context_synchronize", "g4_encode_i32", "g4_decode_i32",
    "g4_encode_f32", "g4_decode_f32", "g4_encode_tiles", "g4_decode_tiles", "g4_encode_arena_bound",
    "g4_fill_terrain", "g4_launch_count", "g4_context_set_timing", "g4_context_set_async", "g4_kernel_time_ms", "g4_codec_supported",
    "g4_crc32c", "g4_tile_records_bound", "g4_pack_tile_records", "g4_unpack_tile_records", "g4_context_order_stream", "g4_decode_tiles_bounded", "g4_predictor_encode", "g4_predictor_encode_int", "g4_predictor_decode",
    "g4_predictor_decode_int", "g4_predictor_tiles", "g4_encode_tile_list", "g4_decode_tile_list", "g4_analyze_tiles",
    "g4_tile_records_bound_multi", "g4_pack_tile_records_multi", "g4_unpack_tile_records_multi",
    "g4_icf_map", "g4_encode_tiles_icf", "g4_decode_tiles_icf", "g4_decode_window",
]


class CodecList(C.Structure):
    _fields_ = [("n_codecs", C.c_int32), ("codec_ids", C.c_int32 * G4_MAX_CODECS)]


class TileRef(C.Structure):
    """g4_tile_ref: where one tile of a tile-list call lives (samples from the base, samples per raster row)."""
    _fields_ = [("offset", C.c_int64), ("pitch", C.c_int64)]


class BandDesc(C.Structure):
    _fields_ = [("elem_type", C.c_int32), ("tile_rows", C.c_int32), ("tile_cols", C.c_int32),
                ("tiles_down", C.c_int32), ("tiles_across", C.c_int32), ("grid_pitch", C.c_int64),
                ("fill_value", C.c_int32), ("reserved", C.c_int32)]


class IcfDesc(C.Structure):
    """g4_icf_desc: the mapping of an integer-coded float element (code = floor((v - offset) * scale + 0.5))."""
    _fields_ = [("scale", C.c_float), ("offset", C.c_float), ("fill_int", C.c_int32), ("fill_value", C.c_float)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "gridfour_b200: %s is missing. The codecs run only as CUDA kernels (no CPU fallback); "
                "build it with `make -C gridfour_b200/csrc`." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.g4_status_string.restype = C.c_char_p
        L.g4_last_error.restype = C.c_char_p
        L.g4_codec_name.restype = C.c_char_p
        L.g4_codec_id_from_name.argtypes = [C.c_char_p]
        L.g4_context_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
        L.g4_context_destroy.argtypes = [C.c_void_p]
        L.g4_context_synchronize.argtypes = [C.c_void_p]
        L.g4_context_order_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.g4_launch_count.argtypes = [C.c_void_p]
        L.g4_launch_count.restype = C.c_uint64
        L.g4_encode_arena_bound.argtypes = [C.POINTER(BandDesc)]
        L.g4_encode_arena_bound.restype = C.c_uint64
        L.g4_encode_i32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                    C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
        L.g4_decode_i32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
        L.g4_encode_f32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                    C.POINTER(C.c_size_t)]
        L.g4_decode_f32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
        L.g4_encode_tiles.argtypes = [C.c_void_p, C.POINTER(CodecList), C.POINTER(BandDesc), C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.POINTER(C.c_uint64)]
        L.g4_decode_tiles.argtypes = [C.c_void_p, C.POINTER(CodecList), C.POINTER(BandDesc), C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]
        L.g4_decode_tiles_bounded.argtypes = [C.c_void_p, C.POINTER(CodecList), C.POINTER(BandDesc), C.c_int, C.c_void_p, C.c_uint64,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.g4_predictor_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int32), C.c_void_p, C.c_size_t,
                                          C.POINTER(C.c_size_t)]
        L.g4_predictor_encode_int.argtypes = L.g4_predictor_encode.argtypes
        L.g4_predictor_decode.argtypes = [C.c_void_p, C.c_int, C.c_int32, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
        L.g4_predictor_decode_int.argtypes = L.g4_predictor_decode.argtypes
        L.g4_predictor_tiles.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(BandDesc), C.c_void_p, C.c_void_p, C.c_uint64,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
        L.g4_encode_tile_list.argtypes = [C.c_void_p, C.POINTER(CodecList), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_uint64)]
        L.g4_decode_tile_list.argtypes = [C.c_void_p, C.POINTER(CodecList), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_uint64,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.g4_analyze_tiles.argtypes = [C.c_void_p, C.POINTER(CodecList), C.POINTER(BandDesc), C.c_int, C.c_void_p, C.c_uint64, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
        L.g4_icf_map.argtypes = [C.c_void_p, C.c_int, C.POINTER(IcfDesc), C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                 C.c_int64]
        L.g4_encode_tiles_icf.argtypes = [C.c_void_p, C.POINTER(CodecList), C.POINTER(BandDesc), C.POINTER(IcfDesc), C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_uint64)]
        L.g4_decode_tiles_icf.argtypes = [C.c_void_p, C.POINTER(CodecList), C.POINTER(BandDesc), C.POINTER(IcfDesc), C.c_int, C.c_void_p,
                                          C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.g4_decode_window.argtypes = [C.c_void_p, C.POINTER(CodecList), C.POINTER(BandDesc), C.POINTER(IcfDesc), C.c_void_p, C.c_uint64,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                       C.c_void_p, C.c_int64, C.c_void_p]
        L.g4_fill_terrain.argtypes =[C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]
        L.g4_context_set_timing.argtypes = [C.c_void_p, C.c_int]
        L.g4_context_set_async.argtypes = [C.c_void_p, C.c_int]
        L.g4_kernel_time_ms.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.g4_kernel_time_ms.restype = C.c_double
        L.g4_crc32c.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.g4_tile_records_bound.argtypes = [C.c_int, C.c_uint64]
        L.g4_tile_records_bound.restype = C.c_uint64
        L.g4_pack_tile_records.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                           C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
        L.g4_unpack_tile_records.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                             C.c_void_p, C.c_void_p]
        L.g4_tile_records_bound_multi.argtypes = [C.c_int, C.c_int, C.c_uint64]
        L.g4_tile_records_bound_multi.restype = C.c_uint64
        L.g4_pack_tile_records_multi.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                                 C.c_int, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
        L.g4_unpack_tile_records_multi.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int, C.c_int,
                                                   C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


class G4Error(Exception):
    def __init__(self, status, where=""):
        self.status = status
        msg = lib().g4_status_string(status).decode()
        if status == G4_ERR_CUDA:
            msg += ": " + lib().g4_last_error().decode()
        super().__init__("%s%s" % (where + ": " if where else "", msg))


class FormatError(G4Error, IOError):
    """Malformed packing -- the reference throws IOException here."""


class ValueChecksumWarning(UserWarning):
    """An LSOP12 packing carries a value checksum that its decoded values do not match.  The reference prints the two
    numbers and returns the values (lsop/LsDecoder12.java:153-158); here the values are returned and this is warned."""


def check(status, where=""):
    if status == G4_OK:
        return
    if status == G4_CHECKSUM_MISMATCH:
        import warnings

        warnings.warn("%s: LSOP12 value checksum mismatch" % (where or "decode"), ValueChecksumWarning, stacklevel=3)
        return
    if status == G4_ERR_FORMAT:
        raise FormatError(status, where)
    raise G4Error(status, where)
