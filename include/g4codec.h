/* g4codec.h -- C ABI of the B200-native GVRS tile-codec library (libg4codec.so).
 *
 * Drop-in boundary for Gridfour's codec plugin API.  Paths cite the reference tree
 * /root/reference/core/src/main/java/org/gridfour/ ("C/").  A Java host binds these symbols through
 * Panama FFM / JNI over pinned direct ByteBuffers (see INTEGRATION.md and java/); every pointer here
 * is a plain address + size, no CUDA or torch types cross the boundary.
 *
 * Reference interfaces replaced:
 *   ICompressionEncoder.encode / encodeFloats          C/compress/ICompressionEncoder.java:61,76
 *   ICompressionDecoder.decode / decodeFloats          C/compress/ICompressionDecoder.java:62,105
 *   CodecMaster.encode / decode (best-of + dispatch)   C/gvrs/CodecMaster.java:142-203
 *   TileElementInt/Float.encode/decode (raw fallback)  C/gvrs/TileElementInt.java:196-219
 *   + the NEW batched encodeTiles / decodeTiles entry the tile cache calls
 *     (natural call sites: C/gvrs/RasterTileCache.java:286-294,339-426, C/gvrs/RecordManager.java:386-515)
 *
 * All compute runs in CUDA kernels for sm_100a.  There is no CPU fallback: every entry point returns
 * G4_ERR_CUDA when no device is usable.
 */
#ifndef G4CODEC_H
#define G4CODEC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define G4_ABI_VERSION 5

/* Status codes.  G4_DECLINED is the Java `null` return of ICompressionEncoder.encode ("codec cannot or
 * should not encode this tile": all-null tile, tile too small for the predictor, singular LSOP matrix).
 * Negative values are errors; the Java shim maps G4_ERR_FORMAT to IOException
 * (C/compress/CodecHuffman.java:166-167, C/compress/CodecDeflate.java:150-152). */
enum {
  G4_OK = 0,
  G4_DECLINED = 1,
  G4_CHECKSUM_MISMATCH = 2, /* decode: the tile's values were delivered, but the value checksum its LSOP12 packing carries
                               does not match them (the reference prints both numbers and carries on, lsop/LsDecoder12.java:153-158) */
  G4_ERR_ARG = -1,      /* bad argument (IllegalArgumentException in the reference) */
  G4_ERR_FORMAT = -2,   /* malformed packing (IOException) */
  G4_ERR_CAPACITY = -3, /* caller's output buffer too small; *out_len holds the size needed */
  G4_ERR_CUDA = -4,     /* no device / CUDA failure; g4_last_error() has the text */
  G4_ERR_UNSUPPORTED = -5
};

/* Codec kinds, named by the identification strings the GVRS file header stores
 * (C/gvrs/GvrsCodecType.java:43-61, C/lsop/LsCodecUtility.java:53). */
enum {
  G4_CODEC_HUFFMAN = 0,       /* "GvrsHuffman"          C/compress/CodecHuffman.java */
  G4_CODEC_DEFLATE = 1,       /* "GvrsDeflate"          C/compress/CodecDeflate.java */
  G4_CODEC_FLOAT = 2,         /* "GvrsFloat"            C/compress/CodecFloat.java */
  G4_CODEC_CANON_HUFFMAN = 3, /* "GvrsCanonicalHuffman" C/compress/canonicalHuffman/CodecCanonHuffman.java */
  G4_CODEC_LSOP12 = 4,        /* "LSOP12"               C/lsop/LsEncoder12.java + LsDecoder12.java */
  G4_CODEC_LSOP08 = 5,        /* "LSOP08"               C/lsop/LsDecoder08.java -- legacy, DECODE ONLY (the reference itself no
                                                         longer registers it, C/lsop/LsCodecUtility.java:73); encode declines */
  G4_CODEC_COUNT = 6
};

/* Options of the LSOP12 encoder (C/lsop/LsEncoder12.java:93-119), OR-ed into a G4_CODEC_LSOP12 entry of a g4_codec_list or
 * into the codec_id of g4_encode_i32, as they belong to the encoder instance in the reference.  Without them LSOP12 encodes
 * as the reference's defaults do: the Deflate alternative on, no value checksum.
 *   G4_LSOP12_NO_DEFLATE      setDeflateEnabled(false): every packing is the canonical-Huffman form (type 2); the Deflate
 *                             alternative (type 1: M32 streams deflated at level 6, kept when its bodies are smaller) is not run.
 *   G4_LSOP12_VALUE_CHECKSUM  setValueChecksumEnabled(true): bit 0x80 of packing[1] is set and the CRC-32C of the tile's values
 *                             (little-endian int32, row-major; for short elements the widened ints, for ICF elements the codes)
 *                             follows the coefficients (type 2, body at byte 59) or [nInit][nInterior] (type 1, body at byte 67).
 * The encode entry points (g4_encode_i32, g4_encode_tiles, g4_encode_tiles_icf, g4_encode_tile_list) honour them; the decode
 * and analyze entry points accept them and ignore them, so that one list serves both directions.  Other bits above the low
 * byte, or option bits on another codec: G4_ERR_ARG.  g4_codec_name and g4_codec_supported take plain ids (an id with option
 * bits has no name and is not supported there). */
#define G4_LSOP12_NO_DEFLATE (1 << 8)
#define G4_LSOP12_VALUE_CHECKSUM (1 << 9)

/* Predictor codes stored in packing[1] (C/compress/PredictorModelType.java:46-63). */
enum { G4_PRED_NONE = 0, G4_PRED_DIFFERENCING = 1, G4_PRED_LINEAR = 2, G4_PRED_TRIANGLE = 3, G4_PRED_DIFF_NULLS = 4 };

/* Sample types of a raster.  G4_ELEM_I16 mirrors TileElementShort (C/gvrs/TileElementShort.java:211-248): samples are
 * widened to int for the codecs with fill_value -> INT4_NULL_CODE, a decoded INT4_NULL_CODE comes back as
 * SHORT_NULL_CODE (-32768), and the raw form is 2 bytes per sample rounded up to a multiple of 4 (TileElement.java:85-93). */
enum { G4_ELEM_I32 = 0, G4_ELEM_F32 = 1, G4_ELEM_I16 = 2, G4_ELEM_ICF = 3 };
enum { G4_MEM_HOST = 0, G4_MEM_DEVICE = 1 };

#define G4_MAX_CODECS 16
#define G4_CODEC_RAW 255 /* per-tile codec byte for "stored raw" (len == 4*nRows*nCols) */

typedef struct g4_context g4_context; /* one CUDA stream + scratch; not shareable between threads */

/* The codec list of a GvrsFileSpecification: position k is the codec index written to packing[0]
 * (C/gvrs/GvrsFileSpecification.java:1576-1631, C/gvrs/CodecMaster.java:153-167). */
typedef struct {
  int32_t n_codecs;
  int32_t codec_ids[G4_MAX_CODECS];
} g4_codec_list;

/* A rectangular band of full-size tiles inside a row-major raster of 4-byte samples.
 * Tile t = tr * tiles_across + tc covers rows [tr*tile_rows, ...) and cols [tc*tile_cols, ...) of the
 * buffer passed as `grid` (whose first sample is the band's upper-left cell). */
typedef struct {
  int32_t elem_type; /* G4_ELEM_I32, G4_ELEM_F32 or G4_ELEM_I16 (G4_ELEM_ICF: the *_icf calls only) */
  int32_t tile_rows, tile_cols;
  int32_t tiles_down, tiles_across;
  int64_t grid_pitch; /* samples per raster row (>= tiles_across*tile_cols); a band may sit inside a wider raster:
                         decode writes the band's columns only, in host and in device memory */
  int32_t fill_value; /* G4_ELEM_I16 encode only: the element's fill value, coded as null */
  int32_t reserved;
} g4_band_desc;

int g4_abi_version(void);
const char* g4_status_string(int status);
const char* g4_last_error(void); /* thread-local text of the last G4_ERR_CUDA */
int g4_device_count(void);

/* "GvrsHuffman" -> G4_CODEC_HUFFMAN ...; -1 for an unknown name. */
int g4_codec_id_from_name(const char* name);
const char* g4_codec_name(int codec_id);

/* device: CUDA ordinal.  cuda_stream: an existing cudaStream_t to launch on (NULL = the context
 * creates its own non-blocking stream). */
int g4_context_create(int device, void* cuda_stream, g4_context** out);
void g4_context_destroy(g4_context* ctx);
int g4_context_synchronize(g4_context* ctx);
/* Stream ordering for G4_MEM_DEVICE buffers that another stream produces or consumes.  A context launches on ITS stream
 * only; device buffers handed to it must be complete on that stream, and results are complete on that stream.  A caller
 * that works on another stream (torch's current stream, a copy stream of the JVM) brackets a call with
 *   g4_context_order_stream(ctx, other, 1);   -- what `other` has queued so far completes before the context's next launch
 *   ... g4_encode_tiles / g4_decode_tiles (G4_MEM_DEVICE) ...
 *   g4_context_order_stream(ctx, other, 0);   -- `other` continues only after what the context has launched so far
 * (events, no host synchronisation).  Passing the context's own stream is a no-op. */
int g4_context_order_stream(g4_context* ctx, void* other_stream, int before);

/* ---- per-tile entry points (exact ICompressionEncoder / ICompressionDecoder semantics) ----------
 * Host buffers.  encode: packing[0] == codec_index; returns G4_DECLINED where the Java codec returns
 * null.  *predictor (optional) receives packing[1]'s predictor code (LSOP12: the compression type). */
int g4_encode_i32(g4_context* ctx, int codec_id, int codec_index, int n_rows, int n_cols, const int32_t* values,
                  uint8_t* out, size_t out_cap, size_t* out_len, int* predictor);
int g4_decode_i32(g4_context* ctx, int codec_id, int n_rows, int n_cols, const uint8_t* packing, size_t len,
                  int32_t* out);
int g4_encode_f32(g4_context* ctx, int codec_id, int codec_index, int n_rows, int n_cols, const float* values,
                  uint8_t* out, size_t out_cap, size_t* out_len);
int g4_decode_f32(g4_context* ctx, int codec_id, int n_rows, int n_cols, const uint8_t* packing, size_t len,
                  float* out);

/* ---- predictor models on their own: IPredictorModel (compress/IPredictorModel.java:42-173) ------------------------------
 * model = G4_PRED_DIFFERENCING / LINEAR / TRIANGLE / DIFF_NULLS.  Host buffers, one tile.
 * g4_predictor_encode      = IPredictorModel.encode:    M32 bytes (capacity 6 * n_rows * n_cols, CodecM32.java:180) + getSeed()
 * g4_predictor_encode_int  = IPredictorModel.encodeInt: residual ints (capacity n_rows * n_cols) + getSeed()
 * g4_predictor_decode(_int)= IPredictorModel.decode / decodeInt.
 * G4_DECLINED where the model returns -1 (Triangle on a one-row tile, the nulls model on a tile of nothing but nulls);
 * G4_ERR_FORMAT for an M32 stream that does not hold exactly the residuals the model needs (the reference reads
 * unchecked, CodecM32.java:321-330). */
int g4_predictor_encode(g4_context* ctx, int model, int n_rows, int n_cols, const int32_t* values, int32_t* seed,
                        uint8_t* m32_out, size_t out_cap, size_t* n_bytes);
int g4_predictor_encode_int(g4_context* ctx, int model, int n_rows, int n_cols, const int32_t* values, int32_t* seed,
                            int32_t* residuals_out, size_t out_cap, size_t* n_residuals);
int g4_predictor_decode(g4_context* ctx, int model, int32_t seed, int n_rows, int n_cols, const uint8_t* m32, size_t n_bytes,
                        int32_t* values_out);
int g4_predictor_decode_int(g4_context* ctx, int model, int32_t seed, int n_rows, int n_cols, const int32_t* residuals,
                            size_t n_residuals, int32_t* values_out);
/* The same for every tile of a band, device buffers: tile t's stream at slots + t * slot_bytes (16-byte aligned; slot_bytes a
 * multiple of 16 and at least 6 * n + 16 for M32 bytes, 4 * n for ints), lens[t] bytes / ints, seeds[t], status[t].
 * decode != 0 runs the inverse (streams -> raster). */
int g4_predictor_tiles(g4_context* ctx, int model, int int_flavour, int decode, const g4_band_desc* band, void* grid,
                       uint8_t* slots, uint64_t slot_bytes, uint32_t* lens, int32_t* seeds, int32_t* status);

/* ---- batched entry points (new) -----------------------------------------------------------------
 * encode: for every tile run every integer (or float) codec of `codecs`, keep the strictly smallest
 * (ties -> lowest index, CodecMaster.encodeSingleThread), store raw little-endian samples when nothing
 * beats 4*n bytes (TileElementInt.encode).  Payloads are packed back to back into `arena` in tile
 * order; offsets[t]/lens[t] locate tile t.  codec_out[t] = winning codec index or G4_CODEC_RAW;
 * predictor_out[t] = packing[1].  All buffers live in `mem_space` (host buffers should be pinned:
 * direct ByteBuffers).  *total_bytes receives the arena bytes used (host value, always).
 * decode: the inverse; len == 4*n means raw (TileElementInt.decode), otherwise packing[0] indexes
 * `codecs`.  status[t] is per tile; the call's return value is the first non-OK tile status or G4_OK. */
int g4_encode_tiles(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space,
                    const void* grid, uint8_t* arena, uint64_t arena_cap, uint64_t* offsets, uint32_t* lens,
                    uint8_t* codec_out, uint8_t* predictor_out, int32_t* status, uint64_t* total_bytes);
int g4_decode_tiles(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space,
                    const uint8_t* arena, const uint64_t* offsets, const uint32_t* lens, void* grid,
                    int32_t* status);

/* g4_decode_tiles for an UNTRUSTED tile directory: arena_len = bytes addressable behind `arena`.  A tile whose
 * offsets[t] + lens[t] leaves the arena, or whose payload is longer than the raw tile, gets status G4_ERR_FORMAT and is
 * never dereferenced.  (g4_decode_tiles itself trusts the directory, e.g. one that g4_unpack_tile_records validated.) */
int g4_decode_tiles_bounded(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space,
                            const uint8_t* arena, uint64_t arena_len, const uint64_t* offsets, const uint32_t* lens,
                            void* grid, int32_t* status);

/* ---- integer-coded float elements (GvrsElementSpecificationIntCodedFloat / GvrsElementIntCodedFloat) -------------------
 * An ICF element stores float values as int codes and its tiles go through the integer codecs untouched, like
 * TileElementInt: raw tiles are the int32 codes (4 bytes per sample), and a fill_int of INT4_NULL_CODE is the null code the
 * predictors know.  The mapping (no reference fixture pins it beyond exactly representable values):
 *   float -> code: NaN -> fill_int; else (int) Math.floor((double)((v - offset) * scale) + 0.5) -- the subtraction and the
 *                  multiplication in float32, correctly rounded and not fused, + 0.5 and floor in double, Java's saturating
 *                  (int) cast.  A finite value whose code is fill_int (-inf with the default fill) reads back as fill_value.
 *   code -> float: fill_int -> fill_value; else (float) code / scale + offset in float32 (a true IEEE division).
 * A NULL descriptor, or a scale that is 0 or not finite: G4_ERR_ARG. */
typedef struct {
  float scale;
  float offset;
  int32_t fill_int;
  float fill_value;
} g4_icf_desc;
/* One rectangle of n_rows x n_cols samples, pitches in samples; to_float != 0 maps codes (int32) to values (float32), else
 * values to codes.  src and dst may be the same buffer.  G4_MEM_DEVICE: one kernel on the context's stream (the result is
 * complete on that stream); G4_MEM_HOST: staged through the device, complete on return. */
int g4_icf_map(g4_context* ctx, int to_float, const g4_icf_desc* icf, int mem_space, int64_t n_rows, int64_t n_cols, const void* src,
               int64_t src_pitch, void* dst, int64_t dst_pitch);
/* g4_encode_tiles / g4_decode_tiles_bounded of an ICF band (band->elem_type == G4_ELEM_ICF; band->fill_value is ignored).
 * Encode maps the float32 band to codes and encodes those (the integer codecs; GvrsFloat in the list is skipped).  Decode
 * decodes the codes into `grid` and maps them to float32 in place, the band's columns only; with g4_context_set_async it
 * only enqueues, as g4_decode_tiles does.  The other band calls reject G4_ELEM_ICF with G4_ERR_ARG. */
int g4_encode_tiles_icf(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, const g4_icf_desc* icf, int mem_space,
                        const float* grid, uint8_t* arena, uint64_t arena_cap, uint64_t* offsets, uint32_t* lens, uint8_t* codec_out,
                        uint8_t* predictor_out, int32_t* status, uint64_t* total_bytes);
int g4_decode_tiles_icf(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, const g4_icf_desc* icf, int mem_space,
                        const uint8_t* arena, uint64_t arena_len, const uint64_t* offsets, const uint32_t* lens, float* grid,
                        int32_t* status);

/* ---- window reads: GvrsElement.readBlock on the device (C/gvrs/GvrsElement.java:298-404) --------------------------------
 * The cells [row0, row0 + n_rows) x [col0, col0 + n_cols) of one element of a raster whose file image is resident on the
 * device, written to out[r * out_pitch + c] (pitch in samples).  Every pointer is a device pointer (host readers keep
 * g4_decode_tiles).  Only the tiles the window touches are decoded.
 *   raster       element type and tile geometry of the WHOLE tile grid (tiles_down x tiles_across tiles; grid_pitch is not
 *                used beyond check_band's rule, tiles_across * tile_cols will do).  G4_ELEM_I32 / F32 / I16, or G4_ELEM_ICF
 *                together with `icf`: the codes are then mapped to float32 values.  To read the codes of an ICF element, pass
 *                G4_ELEM_I32 and no descriptor.
 *   image, image_len, payload_offsets, lens, tile_status
 *                the file image and, in tile-index order, what g4_unpack_tile_records(_multi) returns for the element (one
 *                row of the element-major arrays).  Payloads that leave image_len get G4_ERR_FORMAT, as in
 *                g4_decode_tiles_bounded.
 *   fill_bits    the sample written into the cells of tiles with tile_status G4_DECLINED (absent from the file), as a 32-bit
 *                pattern: float bits for float32 output, the int16 value in the low half for G4_ELEM_I16.
 *   status       one entry per covering tile, in window-tile order (the tile rows and columns the window touches, row-major):
 *                G4_DECLINED for absent tiles (not an error), G4_ERR_FORMAT for a tile whose tile_status is an error or
 *                whose payload is malformed, G4_CHECKSUM_MISMATCH for an LSOP12 value checksum that differs.
 * Returns the first bad status as g4_decode_tiles does, absent tiles not counted (a window of tiles that are all sound or
 * absent returns G4_OK); with g4_context_set_async it only enqueues and returns G4_OK.
 * G4_ERR_ARG for a window that is empty or leaves the tile grid, out_pitch < n_cols, a bad `raster`, or an `icf` for a
 * non-ICF element or with an invalid scale.  A window whose edges lie on tile boundaries is decoded straight into `out`; any
 * other window stages its covering tiles at 4 bytes per sample in device memory the context keeps. */
int g4_decode_window(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* raster, const g4_icf_desc* icf,
                     const uint8_t* image, uint64_t image_len, const uint64_t* payload_offsets, const uint32_t* lens,
                     const int32_t* tile_status, uint32_t fill_bits, int64_t row0, int64_t col0, int64_t n_rows, int64_t n_cols,
                     void* out, int64_t out_pitch, int32_t* status);

/* ---- tile LISTS: scattered tiles of one size (the tile cache's callers) -------------------------------------------------
 * The band calls above take one rectangle of one raster.  A tile cache flushes whatever tiles are dirty, each in its own
 * int[] (gvrs/RasterTileCache.java:253-294, RasterTile.getCompressedPacking :234-256), and a block read lands tiles in a
 * window of the caller's array (gvrs/GvrsElement.java:298-404).  Here every tile has its own reference:
 *   offset = samples from `base` to the tile's cell (0,0), pitch = samples per row of the raster it lives in.
 * `tiles` is a HOST array in both memory spaces; everything else is as in g4_encode_tiles / g4_decode_tiles_bounded
 * (tile t of the call = list position t).  Host rasters are staged by 2-D DMA copies, one per tile -- no host gather.
 * int32 and float32 elements (short elements need the band form: their widening pass works on a rectangle). */
typedef struct g4_tile_ref {
  int64_t offset;
  int64_t pitch;
} g4_tile_ref;
int g4_encode_tile_list(g4_context* ctx, const g4_codec_list* codecs, int elem_type, int tile_rows, int tile_cols, int n_tiles,
                        int mem_space, const void* base, const g4_tile_ref* tiles, uint8_t* arena, uint64_t arena_cap,
                        uint64_t* offsets, uint32_t* lens, uint8_t* codec_out, uint8_t* predictor_out, int32_t* status,
                        uint64_t* total_bytes);
int g4_decode_tile_list(g4_context* ctx, const g4_codec_list* codecs, int elem_type, int tile_rows, int tile_cols, int n_tiles,
                        int mem_space, const uint8_t* arena, uint64_t arena_len, const uint64_t* offsets, const uint32_t* lens,
                        void* base, const g4_tile_ref* tiles, int32_t* status);

/* ---- ICompressionDecoder.analyze (compress/ICompressionDecoder.java:79-92) ------------------------------------------------
 * What CodecHuffman.analyze (:172-199) and CodecDeflate.analyze (:71-106) hand to compress/CodecStats.java:100-155 for
 * one tile: addToCounts(n_bytes, n_symbols, n_bits_overhead) and, from addCountsForM32, the M32 length, the number of
 * distinct M32 bytes and the first-order entropy of the tile's M32 stream (bits per byte).  status: G4_OK, G4_DECLINED for
 * tiles that carry no M32 statistics (raw tiles, the other codecs), G4_ERR_FORMAT for a malformed packing. */
typedef struct g4_tile_stats {
  int32_t codec_kind;       /* G4_CODEC_* of the packing, -1 for a raw tile */
  int32_t predictor;        /* packing[1] */
  uint32_t n_bytes;         /* packing length - 10 */
  uint32_t n_symbols;       /* n_rows * n_cols */
  uint32_t n_bits_overhead; /* HuffmanDecoder.getBitsInTreeCount(); 0 for CodecDeflate */
  uint32_t n_m32;
  uint32_t observed;        /* distinct M32 byte values */
  int32_t status;
  double entropy;
} g4_tile_stats;
/* Every tile of a batch (arguments as in g4_decode_tiles_bounded).  pair_counts (optional, same memory space, caller-zeroed):
 * [2][5][65536] uint64 successor counts CodecStats.sB -- first index 0 = CodecHuffman, 1 = CodecDeflate, second = the
 * predictor code -- which the calls ADD to (CodecStats.getH2 :133-165 works on these; sA is the column sum of sB). */
int g4_analyze_tiles(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space, const uint8_t* arena,
                     uint64_t arena_len, const uint64_t* offsets, const uint32_t* lens, g4_tile_stats* stats,
                     uint64_t* pair_counts);

/* Upper bound of the arena bytes g4_encode_tiles can produce for a band (4*n per tile). */
uint64_t g4_encode_arena_bound(const g4_band_desc* band);


/* ---- GVRS tile records: the wire format either side of the codec path (SURVEY section 8f, row 1) -----------------------
 * A record is [size:int32 LE][type:uint8][0,0,0] content, zero padding, [crc32c:int32 LE]; size is a multiple of 8 and
 * counts everything (C/gvrs/RecordManager.java:70-78,137-139,161-204).  A tile record (type 2) of a one-element raster
 * holds [tileIndex:int32][len:int32][len bytes] (RecordManager.writeTile :386-490; len == 4*nRows*nCols means raw samples,
 * RecordManager.readTile :492-516).  The tile directory stores the position of the CONTENT (record position + 8) divided
 * by 8 (C/gvrs/TileDirectory.java:121-146).  mem_space says where data / arena / records / image live; the small
 * per-tile arrays (offsets, lens, positions, status) live in the same space. */

/* CRC-32C of n byte ranges data[offsets[i] .. +sizes[i]) (C/util/GridfourCRC32C.java:156-163: Castagnoli polynomial,
 * reflected, initial value and final xor 0xffffffff -- what RecordManager.fileSpaceFinishRecord stores). */
int g4_crc32c(g4_context* ctx, int mem_space, const uint8_t* data, const uint64_t* offsets, const uint32_t* sizes, int n,
              uint32_t* crc_out);

/* Upper bound of the record bytes g4_pack_tile_records writes for n_tiles payloads of payload_bytes in total. */
uint64_t g4_tile_records_bound(int n_tiles, uint64_t payload_bytes);

/* Frames the payloads of a batch (what g4_encode_tiles returned) as consecutive tile records, the first one at file
 * position base_pos (a multiple of 8).  tile_index may be NULL: record t then carries first_tile_index + t.  checksum != 0
 * computes the CRC-32C of every record, otherwise the field stays zero like in the reference.  content_pos[t] receives the
 * file position the tile directory has to store for tile t; *total_bytes the number of record bytes written. */
int g4_pack_tile_records(g4_context* ctx, int mem_space, const uint8_t* arena, const uint64_t* offsets, const uint32_t* lens,
                         const int32_t* tile_index, int first_tile_index, int n_tiles, int checksum, uint64_t base_pos,
                         uint8_t* records, uint64_t records_cap, uint64_t* content_pos, uint64_t* total_bytes);

/* Inverse: image is a GVRS file (or a part of one: content_pos is relative to image) of image_len bytes, content_pos[t]
 * the directory position of tile t (0 = tile absent -> status G4_DECLINED, len 0).  Checks every record (type, sizes,
 * bounds and, with checksum != 0, the CRC-32C) and returns payload_offsets / lens in the form g4_decode_tiles takes with
 * `image` as its arena.  A damaged record gives status G4_ERR_FORMAT for that tile; the call itself still succeeds.  A record
 * whose CRC differs also gets G4_ERR_FORMAT here (g4_unpack_tile_records_multi tells it apart as G4_CHECKSUM_MISMATCH). */
int g4_unpack_tile_records(g4_context* ctx, int mem_space, const uint8_t* image, uint64_t image_len, const uint64_t* content_pos,
                           int n_tiles, int checksum, uint64_t* payload_offsets, uint32_t* lens, int32_t* status);

/* ---- tile records of rasters with several elements per tile (RecordManager.writeTile / readTile :386-516) ------------------
 * content = [tileIndex:int32] then, for each element e in specification order, [len_e:int32][len_e bytes]; the record size
 * is multipleOf8(12 + 4 + sum_e(4 + len_e)).  Element e's payload is what g4_encode_tiles returned for that element (a codec
 * packing, or the raw tile at the element's standard size).  With n_elements == 1 these calls write and read exactly the
 * records of g4_pack_tile_records / g4_unpack_tile_records.  n_elements outside 1..G4_MAX_ELEMENTS: G4_ERR_UNSUPPORTED. */
#define G4_MAX_ELEMENTS 64
/* Upper bound of the record bytes g4_pack_tile_records_multi writes for n_tiles tiles with payload_bytes in total (0 for
 * arguments out of range). */
uint64_t g4_tile_records_bound_multi(int n_tiles, int n_elements, uint64_t payload_bytes);
/* arenas / offsets / lens: HOST arrays of n_elements pointers (like g4_tile_ref); the buffers they point to live in mem_space.
 * Element e of tile t is arenas[e][offsets[e][t] .. + lens[e][t]), at any alignment.  Host buffers are staged: for each
 * element its range [0, max_t(offsets[e][t] + lens[e][t])) is copied.  The other arguments and results are those of
 * g4_pack_tile_records, including G4_ERR_CAPACITY with the needed size in *total_bytes. */
int g4_pack_tile_records_multi(g4_context* ctx, int mem_space, int n_elements, const uint8_t* const* arenas,
                               const uint64_t* const* offsets, const uint32_t* const* lens, const int32_t* tile_index,
                               int first_tile_index, int n_tiles, int checksum, uint64_t base_pos, uint8_t* records,
                               uint64_t records_cap, uint64_t* content_pos, uint64_t* total_bytes);
/* Inverse.  payload_offsets / lens: n_elements x n_tiles, ELEMENT-major (element e of tile t at e * n_tiles + t), so that row e
 * feeds g4_decode_tiles directly with `image` as the arena.  status[t]: G4_OK; G4_DECLINED for content_pos 0 (tile absent);
 * G4_ERR_FORMAT for a damaged record (misaligned or out-of-image position, type, size, a len with bit 31 set, or a chain
 * that runs into the checksum field); G4_CHECKSUM_MISMATCH, with checksum != 0, for a sound record whose CRC differs.  Every
 * tile whose status is not G4_OK gets offset 0 and length 0 for every element.  The call itself still succeeds. */
int g4_unpack_tile_records_multi(g4_context* ctx, int mem_space, int n_elements, const uint8_t* image, uint64_t image_len,
                                 const uint64_t* content_pos, int n_tiles, int checksum, uint64_t* payload_offsets,
                                 uint32_t* lens, int32_t* status);

/* ---- benchmark support --------------------------------------------------------------------------
 * Fills a device raster with the synthetic fractal terrain of include/g4terrain.h
 * (rows [row0,row0+n_rows) x cols [col0,col0+n_cols) of the virtual global grid). */
int g4_fill_terrain(g4_context* ctx, int elem_type, uint64_t seed, int64_t row0, int64_t col0, int64_t n_rows,
                    int64_t n_cols, void* device_out);
/* Kernel launches issued through this context since creation (bench.py's gpu_launches claim). */
uint64_t g4_launch_count(const g4_context* ctx);
/* Per-kernel device timing: when enabled, every codec kernel launch is bracketed by CUDA events on the
 * context's stream.  g4_kernel_time_ms returns the duration of the most recent launch of the decode
 * (direction 0) or encode (direction 1) kernel of `codec_kind` (G4_CODEC_COUNT = raw copy); < 0 if none. */
int g4_context_set_timing(g4_context* ctx, int enabled);
/* Pipelined device calls.  By default g4_decode_tiles / g4_decode_tile_list with G4_MEM_DEVICE wait for the batch and
 * return the first failing tile's status.  With `enabled` they only ENQUEUE the batch on the context's stream and return
 * G4_OK: `status[]` (device memory) holds the per-tile results once the stream has run (g4_context_synchronize), so a tile
 * cache can keep several windows of tiles in flight (C/gvrs/RasterTileCache.java:339-426 reads ahead the same way with its
 * TileDecompressionAssistant).  Host-memory calls are not affected. */
int g4_context_set_async(g4_context* ctx, int enabled);
/* 1 when the CUDA kernels for codec_id exist for direction (0 = decode, 1 = encode), else 0. */
int g4_codec_supported(int codec_id, int direction);
double g4_kernel_time_ms(g4_context* ctx, int direction, int codec_kind);

#ifdef __cplusplus
}
#endif
#endif
