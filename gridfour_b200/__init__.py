"""gridfour_b200 -- GVRS tile codecs as sm_100a CUDA kernels behind Gridfour's codec plugin API.

Host-side mirror (Python, over the C ABI in include/g4codec.h) of the reference's Java interfaces:
ICompressionEncoder / ICompressionDecoder, the codec classes, GvrsFileSpecification.addCompressionCodec and
CodecMaster, plus the new batched encodeTiles / decodeTiles entry.  See DESIGN.md and INTEGRATION.md.
"""
from .codecs import (  # noqa: F401
    CodecCanonHuffman, CodecDeflate, CodecFloat, CodecHuffman, CodecMaster, CodecSpecification, Context,
    ICompressionDecoder, ICompressionEncoder, IntCodedFloat, LsDecoder08, LsDecoder12, LsEncoder08, LsEncoder12, TileBatch,
    INT4_NULL_CODE,
)
from ._lib import FormatError, G4Error, ValueChecksumWarning  # noqa: F401
from . import gvrs  # noqa: F401
from .sharding import gather_layout, record_offsets, shard_tile_rows, tile_content, tile_record_is_compressed  # noqa: F401
from .predictors import (  # noqa: F401
    IPredictorModel, PredictorModelDifferencing, PredictorModelDifferencingWithNulls, PredictorModelLinear, PredictorModelTriangle,
    PredictorModelType,
)
from .tilecache import RasterTileCache  # noqa: F401
from .stats import CodecStats, analyze_tiles  # noqa: F401
