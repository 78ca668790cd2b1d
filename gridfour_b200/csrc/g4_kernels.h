// g4_kernels.h -- kernel argument blocks and launch entry points shared by the codec translation units.
#pragma once
#include <cstddef>
#include <cstdint>
#include <atomic>
#include <cuda_runtime.h>
#include "../../include/g4codec.h"
#include "g4_device.cuh"

namespace g4 {

// cudaFuncSetAttribute is per DEVICE: `done` holds one bit per device ordinal.  Setting an attribute twice is harmless, so
// two threads racing on the same device need no lock.
template <class Fn>
inline cudaError_t once_per_device(std::atomic<uint64_t>& done, Fn set) {
  int d = 0;
  cudaGetDevice(&d);
  const uint64_t bit = 1ull << (d & 63);
  if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
  const cudaError_t e = set();
  if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
  return e;
}

struct DeflateBlocks;  // g4_deflate_enc.cuh

// One candidate-encoder launch: every tile of the band is encoded by ONE codec into its own fixed-size
// slot (slot t at slots + t*slotBytes, 16-byte aligned).  lens[t] = packing length (0 = declined).
struct EncodeArgs {
  BandEx band;
  void* grid;           // device raster (band upper-left cell)
  uint8_t* slots;
  size_t slotBytes;
  uint32_t* lens;
  uint8_t* preds;       // packing[1] of the candidate
  int32_t* status;      // G4_OK / G4_DECLINED / error
  int* counter;         // persistent-CTA work counter (zeroed before launch)
  int codecIndex;       // list position of this codec == packing[0]
  uint8_t* scratch;     // per-CTA scratch (codec specific)
  size_t scratchStride;
  const uint32_t* valueCrc;  // LSOP12: per-tile value checksum to store in the header (launch_lsop_value_crc), or null
};

// One decoder launch over the tiles of one codec kind: list[0..*listCount) are tile indices.
struct DecodeArgs {
  BandEx band;
  void* grid;
  const uint8_t* arena;
  const uint64_t* offsets;
  const uint32_t* lens;
  const int* list;
  const int* listCount;
  int32_t* status;
  int* counter;
  uint8_t* scratch;     // per-CTA scratch (M32 bytes etc.), blockIdx.x * scratchStride
  size_t scratchStride;
  int rawShorts;        // raw tiles hold 2-byte samples (TileElementShort): widen them into the int32 raster
  uint32_t* lsopCks;    // LSOP12: [tile][2] = {packing carries a value checksum, its value}; zeroed before the launch set, or null
};

struct SelectArgs {
  int nTiles, nCand;
  uint32_t rawLen;              // 4 * tile_rows * tile_cols
  const uint32_t* candLens;     // [nCand][nTiles]
  const uint8_t* candPreds;     // [nCand][nTiles]
  const int32_t* candStatus;    // [nCand][nTiles]
  int candIndex[G4_MAX_CODECS]; // codec list position of candidate c
  uint32_t* lens;               // out: payload length per tile
  uint8_t* codecOut;
  uint8_t* predOut;
  int* src;                     // out: winning candidate (-1 = raw)
  int32_t* status;
};

struct CompactArgs {
  BandEx band;
  void* grid;
  const uint8_t* slots[G4_MAX_CODECS];
  size_t slotBytes;
  const uint32_t* lens;
  const uint64_t* offsets;
  const int* src;
  uint8_t* arena;
  uint64_t arenaCap;
  int32_t* status;
  int rawShorts;          // TileElementShort: raw tiles take 2 bytes per sample, narrowed from the int32 staging raster `grid`
  int32_t fill16;         // ... with INT4_NULL_CODE -> the element's fill value (the inverse of window_load_kernel's widening)
};

struct ClassifyArgs {
  int nTiles;
  int elemType;
  uint32_t rawLen;
  g4_codec_list codecs;
  const uint8_t* arena;
  uint64_t arenaLen;  // bytes addressable behind `arena` (UINT64_MAX = the caller vouches for the directory)
  const uint64_t* offsets;
  const uint32_t* lens;
  int* lists;    // [G4_CODEC_COUNT + 1][nTiles]
  int* counts;   // [G4_CODEC_COUNT + 1], zeroed before launch
  int32_t* status;
};

// zlib streams of a band: stream j reads inBuf + inOff[j] (inLen[j] bytes, 0 = skip) and writes at most
// inLen[j] + capExtra bytes to outBuf + inOff[j] + 112*j; outLen[j] = bytes written (g4_deflate_encode.cu).
struct StreamArgs {
  const uint8_t* inBuf;
  const uint64_t* inOff;
  const uint32_t* inLen;
  uint8_t* outBuf;
  uint32_t* outLen;
  int nStreams;
  int capExtra;  // 118 CodecDeflate (:206-210), 128 CodecFloat / LSOP12
  int level;     // 6 or 9
  void* work;    // nWorkers * deflate_work_bytes()
  int* counter;  // zeroed before launch
  int bigOnly;   // 1: only streams longer than deflate_staged_max() (the staged kernels take the rest)
};

// Staged zlib encode of the streams [jBegin, jEnd) that are at most deflate_staged_max() bytes long
// (g4_deflate_enc.cuh, "Staged form").  The per-position scratch arrays are indexed by inOff[j] - baseOff + position.
struct StagedArgs {
  const uint8_t* inBuf;
  const uint64_t* inOff;
  const uint32_t* inLen;
  uint8_t* outBuf;
  uint32_t* outLen;
  int jBegin, jEnd;
  uint64_t baseOff;
  uint16_t* sorted;   // positions ordered by (hash, position)
  uint16_t* rank;     // number of earlier positions in the slot's hash bucket
  uint32_t* table;    // per position: longest match with the full chain (def_pack_match; bit 31: tableQ differs)
  uint32_t* tableQ;   // per position, written only where it differs: longest match with the quarter chain
  uint32_t maxLen;    // longest staged stream of the chunk (sizes the match kernel's shared-memory table)
  int lazy;           // deep levels: the sort also writes position -> slot (into `rank`), one warp per stream parses and
                      // searches only where zlib would (symbols then live in the table arrays)
  DeflateBlocks* blocks;  // per stream of the chunk: block boundaries (decide kernel -> emit kernel), deflate_blocks_bytes() each
  int capExtra, level;
  int* counters;      // 4 ints, zeroed before launch
};

cudaError_t launch_fill_terrain(int elemType, uint64_t seed, int64_t row0, int64_t col0, int64_t nRows, int64_t nCols, void* out,
                                cudaStream_t s);
cudaError_t launch_select(const SelectArgs& a, cudaStream_t s);
cudaError_t launch_offsets(const uint32_t* lens, uint64_t* offsets, int nTiles, uint64_t* total, cudaStream_t s);
cudaError_t launch_compact(const CompactArgs& a, int nTiles, cudaStream_t s);
cudaError_t launch_classify(const ClassifyArgs& a, cudaStream_t s);
cudaError_t launch_raw_decode(const DecodeArgs& a, int nTiles, cudaStream_t s);
// TileElementShort (gvrs/TileElementShort.java:236-248): the decoded int32 raster -> int16 (the encode side widens in
// window_load_kernel)
cudaError_t launch_narrow_i16(const int32_t* src, int16_t* dst, int64_t dstPitch, int64_t rows, int64_t cols, cudaStream_t s);
// Integer-coded float elements: float32 <-> int32 codes over a pitched rectangle (pitches in samples; src may equal dst).
// toFloat != 0 runs icf_to_float_kernel (codes -> values), else icf_to_int_kernel (values -> codes).
struct IcfMap {
  float scale, offset;
  int32_t fillInt;
  float fillValue;
};
cudaError_t launch_icf_map(int toFloat, const void* src, int64_t srcPitch, void* dst, int64_t dstPitch, int64_t rows, int64_t cols,
                           const IcfMap& m, cudaStream_t s);

// Window writes (g4_encode_window, and the staging of every short encode): one pass from the caller's n_rows x n_cols raster
// (any pitch) into the int32 staging raster of the covering tile grid (rows x cols cells, pitch dstPitch).  Cells inside the
// raster are converted by `mode`, the cells outside it get the margin sample fillBits converted by the same rule, so that a
// margin cell encodes exactly as if the caller had padded the raster with that sample.
enum { kLoadCopy32 = 0, kLoadWiden16 = 1, kLoadIcfCode = 2 };  // how a source sample becomes a staged int32
struct WindowLoad {
  const void* src;        // int32 / float32 / int16 samples
  int64_t srcPitch;       // samples per source row
  int64_t nRows, nCols;   // the source raster
  int32_t* dst;           // staging raster
  int64_t dstPitch;       // samples per staging row
  int64_t rows, cols;     // staged cells (rows >= nRows, cols >= nCols)
  uint32_t fillBits;      // margin sample as a 32-bit pattern of the source type (the int16 in the low half for kLoadWiden16)
  int32_t fill16;         // kLoadWiden16: the element's fill value, staged as INT4_NULL_CODE (TileElementShort.java:213-220)
  int mode;               // kLoad*
  IcfMap icf;             // kLoadIcfCode
};
cudaError_t launch_window_load(const WindowLoad& a, cudaStream_t s);

// Window reads (g4_decode_window): the tiles tr0.. x tc0.. (nTd x nTa, "window tiles" w = wr * nTa + wc) of a raster whose
// per-tile arrays are in tile-index order.  The gather copies the window tiles' payload locations into window order; a tile
// whose status is not G4_OK gets offset 0 and length 0 (classify_kernel then keeps it out of every decoder list) and, when
// it is G4_DECLINED, absent[w] = 1.
cudaError_t launch_window_gather(const uint64_t* offsets, const uint32_t* lens, const int32_t* tileStatus, int tilesAcross, int tr0,
                                 int tc0, int nTd, int nTa, uint64_t* offW, uint32_t* lenW, uint8_t* absentW, cudaStream_t s);
enum { kWindowCopy32 = 0, kWindowNarrow16 = 1, kWindowIcfFloat = 2 };  // how a decoded int32 sample becomes an output sample
struct WindowStore {
  const int32_t* stage;   // the decoded window tiles (int32 / float32 bits / ICF codes); null: decoded in place (tile-aligned)
  int64_t stagePitch;     // samples per staging row
  int64_t sr0, sc0;       // staging cell of output cell (0, 0)
  int64_t rows, cols;     // output rectangle
  void* out;
  int64_t outPitch;       // samples per output row
  int R, C, nTa, nW;      // tile size, window tiles across, window tiles
  const uint8_t* absent;  // [nW] from launch_window_gather
  int32_t* status;        // [nW]: absent tiles get G4_DECLINED
  uint32_t fillBits;      // output sample of absent tiles (the low 16 bits for kWindowNarrow16)
  int mode;               // kWindow*
  IcfMap icf;             // kWindowIcfFloat
};
// stage != null: one pass stage -> out (crop, narrow / ICF map, fill of absent tiles).  stage == null: the window tiles were
// decoded straight into out; only the absent ones are filled.
cudaError_t launch_window_store(const WindowStore& a, int smCount, cudaStream_t s);

// Point and block reads (g4_decode_points, g4_decode_blocks): the blockRows x blockCols block at (rows[i], cols[i]) of the
// raster for each of n blocks; a point is a 1 x 1 block.  The mark pass sets flag[t] for every tile a block covers
// (info[0] = 1 for a block not wholly inside the raster); the compaction pass, one CTA, scans the flags in tile-index order:
// the k-th touched tile t gets slot[t] = k, tilesOut[k] = t, its payload location and absent flag as launch_window_gather
// gives them, and info[1] = K.  The compaction leaves every flag zero again, so the flag array (nTiles rounded up to 16
// bytes, zero padded) is zero between calls; info[0] is cleared by the caller that reads it set.
struct PointArgs {
  const int64_t* rows;
  const int64_t* cols;
  int64_t n;
  int64_t rasterRows, rasterCols;  // blocks must lie in [0, rasterRows) x [0, rasterCols)
  int R, C, tilesAcross, nTiles;
  uint8_t* flag;                   // [nTiles rounded up to 16]
  int32_t* info;                   // [0] a point outside the raster, [1] K
  int32_t* slot;                   // [nTiles]: valid for touched tiles
  const uint64_t* offsets;         // per tile of the raster, tile-index order
  const uint32_t* lens;
  const int32_t* tileStatus;
  int32_t* tilesOut;               // [K] touched tiles, ascending
  uint64_t* offK;                  // [K] payload locations in slot order (zero-length for tiles not G4_OK)
  uint32_t* lenK;
  uint8_t* absentK;                // [K] 1 for G4_DECLINED
  int64_t blockRows, blockCols;    // 1 x 1 for points
  int coverTd, coverTa;            // most tile rows / columns one block can cover (1 x 1 for points)
};
cudaError_t launch_point_mark(const PointArgs& a, int smCount, cudaStream_t s);
cudaError_t launch_point_compact(const PointArgs& a, cudaStream_t s);
// w.stage holds the K touched tiles decoded as a K x 1 band (tile k at k * R * C, pitch C); w.absent / w.status are in slot
// order (w.nW = K).  out[i] = the converted sample of point i, or the fill sample for an absent tile; absent tiles' status
// becomes G4_DECLINED.
cudaError_t launch_point_store(const PointArgs& p, const WindowStore& w, int smCount, cudaStream_t s);
// The same staging and slots; out + i * blockRows * blockCols = block i, rows contiguous, converted and filled as above.
cudaError_t launch_block_store(const PointArgs& p, const WindowStore& w, int smCount, cudaStream_t s);

// ---- codec kernels -----------------------------------------------------------------------------
// Host-side launchers (defined next to their kernels).  nCtas persistent CTAs of kThreads threads.
cudaError_t launch_huffman_encode(const EncodeArgs& a, int nCtas, cudaStream_t s);
// fused fast path of the legacy Huffman decoder (g4_huff2.cuh): per-context scratch
struct HuffFusedScratch {
  uint32_t* spill;   // huffman2_spill_bytes(smCount)
  uint8_t* trees;    // huffman2_tree_bytes(nTiles): per-tile tree records of huffman2_tree_kernel
  int* defer;        // nTiles ints: tiles left to huffman_decode_kernel
  int* counters;     // [0] defer count, [1] tile counter of the second kernel; both zero before the launch
  int smCount;
};
size_t huffman2_spill_bytes(int smCount);
size_t huffman2_tree_bytes(int nTiles);
cudaError_t launch_huffman_decode(const DecodeArgs& a, int nCtas, cudaStream_t s, const HuffFusedScratch& fused, int* launches);
cudaError_t launch_canon_decode(const DecodeArgs& a, int nCtas, cudaStream_t s);
cudaError_t launch_canon_encode(const EncodeArgs& a, int nCtas, cudaStream_t s);  // needs 32 KB scratch per CTA
cudaError_t launch_lsop_encode(const EncodeArgs& a, int nCtas, cudaStream_t s);   // needs 32 KB scratch per CTA
// region: HBM staging for inflated bytes, one slot of regionStride bytes per list position
cudaError_t launch_deflate_decode(const DecodeArgs& a, uint8_t* region, size_t regionStride, int nCtas, int nTilesUpper,
                                  cudaStream_t s);
cudaError_t launch_float_decode(const DecodeArgs& a, uint8_t* region, size_t regionStride, int nCtas, int nTilesUpper,
                                cudaStream_t s);
// coef: [nTiles][12] floats of device scratch; nTilesUpper bounds the number of LSOP tiles in the list
// defer: nTilesUpper ints; deferCounters: 4 zeroed ints (deferred-tile count, work counters of the general kernel, of the
// text kernel and of the fast path's wavefront kernel)
// meta: nTilesUpper * lsop_meta_bytes() bytes (interior code lengths + text position handed from kernel H to kernel T)
size_t lsop_meta_bytes();
// LSOP08, the legacy 8-coefficient codec (decode only): entropy stage + initializers, then the wavefront
cudaError_t launch_lsop08_decode(const DecodeArgs& a, float* coef, int nCtas, int nTilesUpper, cudaStream_t s);


// LSOP12 decode, fast path (g4_lsop_fast.cu): byte hand-over between the text kernel and a TMA-fed wavefront kernel.
struct LsopFastGeom {
  int R, C;
  int W;          // strip width in columns: 4, 8 or 16 (C is a multiple of W)
  int logW;
  int tilesPerWarp;  // wavefront tiles per warp: 2 when nStrips <= 16 (each 16-lane half of the warp decodes its own
                     // tile), else 1
  int nStrips;    // lanes of a wavefront tile in use: strip k = columns 2 + k W .. 2 + k W + W - 1; ceil((C - 2) / W) <= 32
                  // (<= 16 with two tiles per warp)
  int P;          // bytes per row of the residual image = nStrips * W
  int nSteps;     // wavefront steps = R - 2 + nStrips - 1 (lane k works on row s - k + 2 at step s)
  int chunkRows;  // image rows per bulk copy of the wavefront kernel = 128 / W (chunk = chunkRows * P <= 4096 bytes;
                  // <= 2048 with two tiles per warp, which share one 4096-byte ring stage)
  int nChunks;
  int tileBytes;  // nChunks * chunkRows * P: the image one tile writes
  int tilePitch;  // bytes between the images of consecutive tiles (a multiple of 128)
  int wide;       // 256-bit raster stores
};
struct LsopFastArgs {
  DecodeArgs a;
  float* coef;        // [nTiles][12]
  uint8_t* meta;      // [nTiles][lsop_meta_bytes()]
  int4* side;         // [nTiles][R]: {v[r][0], v[r][1], D2[r], D1[r]}
  uint32_t* exc;      // [nTiles][128]: residuals that are no byte
  uint8_t* resid;     // residual scratch (lsop_fast_resid_bytes)
  uint8_t* textStage; // spill words behind the staging slots of the text kernel, one area per persistent CTA (lsop_fast_stage_bytes)
  int* defer;         // tiles for the general kernels
  int* deferCount;
  LsopFastGeom g;
};
bool lsop_fast_geometry(const g4_band_desc& band, const void* grid, LsopFastGeom* out);
size_t lsop_fast_side_bytes(const LsopFastGeom& g, int nTiles);
size_t lsop_fast_exc_bytes(int nTiles);
size_t lsop_fast_stage_bytes(int smCount);
size_t lsop_fast_resid_bytes(const LsopFastGeom& g, int nTiles);
cudaError_t launch_lsop_decode_fast(const LsopFastArgs& A, int nTilesUpper, int smCount, int* textCounter, cudaStream_t s, int* launches);
// fast: scratch of the fast path (side / exc / resid / g filled in), or null -> the round-1 kernels only
cudaError_t launch_lsop_decode(const DecodeArgs& a, float* coef, uint8_t* meta, int* defer, int* deferCounters, int nCtas,
                               int nTilesUpper, cudaStream_t s, int* launches, const LsopFastArgs* fast = nullptr, int smCount = 148);

// ICompressionDecoder.analyze (g4_analyze.cu): per-tile M32 statistics of CodecHuffman / CodecDeflate packings.
struct AnalyzeArgs {
  int nTiles;
  uint32_t nCells;    // tile_rows * tile_cols
  uint32_t rawLen;
  g4_codec_list codecs;
  const uint8_t* arena;
  uint64_t arenaLen;
  const uint64_t* offsets;
  const uint32_t* lens;
  uint8_t* scratch;   // per-CTA M32 scratch, blockIdx.x * scratchStride (6 * nCells + 64, 16-byte aligned)
  size_t scratchStride;
  g4_tile_stats* stats;        // [nTiles]
  unsigned long long* pairs;   // [2 codecs][5 predictor codes][65536] successor counts (CodecStats.sB), or null
};
cudaError_t launch_analyze(const AnalyzeArgs& a, int nCtas, cudaStream_t s);

// Predictor models on their own (g4_predictor.cu): IPredictorModel.encode / decode / encodeInt / decodeInt over a band.
struct PredictorArgs {
  BandEx band;
  void* grid;          // int32 raster: source of encode, destination of decode
  int model;           // G4_PRED_DIFFERENCING .. G4_PRED_DIFF_NULLS
  int intFlavour;      // 1: residual ints (encodeInt / decodeInt), 0: M32 bytes
  uint8_t* slots;      // tile t at slots + t * slotBytes (16-byte aligned; M32 input padded by 16 readable bytes)
  size_t slotBytes;
  uint32_t* lens;      // bytes / ints per tile
  int32_t* seeds;
  int32_t* status;
};
cudaError_t launch_predictor(const PredictorArgs& a, int decode, int nCtas, cudaStream_t s);

// ---- zlib-stream encode stages (g4_deflate_encode.cu, g4_lsop.cu) ------------------------------------------------
size_t deflate_work_bytes();
size_t deflate_blocks_bytes();
uint32_t deflate_staged_max();
cudaError_t launch_deflate_staged(const StagedArgs& a, int smCount, cudaStream_t s);
cudaError_t launch_stream_offsets(const uint32_t* inLen, uint64_t* inOff, int nStreams, uint64_t* total, cudaStream_t s);
cudaError_t launch_deflate_streams(const StreamArgs& a, int nWorkers, cudaStream_t s);
cudaError_t launch_deflate_m32_size(const EncodeArgs& a, uint32_t* inLen, int nCtas, cudaStream_t s);
cudaError_t launch_deflate_m32_write(const EncodeArgs& a, const uint32_t* inLen, const uint64_t* inOff, uint8_t* inBuf, int nCtas,
                                     cudaStream_t s);
cudaError_t launch_deflate_pick(const EncodeArgs& a, const uint32_t* inLen, const uint64_t* inOff, const uint8_t* outBuf,
                                const uint32_t* outLen, int nCtas, cudaStream_t s);
cudaError_t launch_float_plane_size(int nTiles, uint32_t n, uint32_t* inLen, cudaStream_t s);
cudaError_t launch_float_plane_write(const EncodeArgs& a, const uint64_t* inOff, uint8_t* inBuf, int nCtas, cudaStream_t s);
cudaError_t launch_float_pick(const EncodeArgs& a, const uint64_t* inOff, const uint8_t* outBuf, const uint32_t* outLen, int nCtas,
                              cudaStream_t s);
// LSOP12 Deflate alternative (LsEncoder12.java:170-218): streams 2t (initializers) and 2t+1 (interior)
cudaError_t launch_lsop_m32_size(const EncodeArgs& a, uint32_t* inLen, int nCtas, cudaStream_t s);
cudaError_t launch_lsop_m32_write(const EncodeArgs& a, const uint32_t* inLen, const uint64_t* inOff, uint8_t* inBuf, int nCtas,
                                  cudaStream_t s);
cudaError_t launch_lsop_pick(const EncodeArgs& a, const uint32_t* inLen, const uint64_t* inOff, const uint8_t* outBuf,
                             const uint32_t* outLen, int nCtas, cudaStream_t s);

// ---- GVRS tile records (g4_records.cu) --------------------------------------------------------------------------------
cudaError_t launch_crc32c(const uint8_t* data, const uint64_t* offsets, const uint32_t* sizes, int n, uint32_t* out, int storeAtEnd,
                          cudaStream_t s);
cudaError_t launch_record_layout(const uint32_t* lens, int n, uint64_t basePos, uint64_t* contentPos, uint64_t* crcOff, uint32_t* crcLen,
                                 uint64_t* total, cudaStream_t s);
cudaError_t launch_record_pack(const uint8_t* arena, const uint64_t* offsets, const uint32_t* lens, const int32_t* tileIndex,
                               int firstTileIndex, int n, const uint64_t* crcOff, const uint32_t* crcLen, uint8_t* records, int nCtas,
                               cudaStream_t s);
cudaError_t launch_record_unpack(const uint8_t* image, uint64_t imageLen, const uint64_t* contentPos, int n, uint64_t* payloadOff,
                                 uint32_t* lens, uint64_t* crcOff, uint32_t* crcLen, uint32_t* storedCrc, int32_t* status, cudaStream_t s);
// LSOP12 value checksum (LsDecoder12.java:153-158): CRC-32C of every decoded tile whose packing carries one, compared with the
// stored value; a mismatch leaves status G4_CHECKSUM_MISMATCH (the values stay delivered: the reference only prints).
cudaError_t launch_lsop_value_checksum(const DecodeArgs& a, int nTilesUpper, cudaStream_t s);
// LSOP12 encode with the value checksum: crc[t] = CRC-32C of tile t's values, every tile of a.band
cudaError_t launch_lsop_value_crc(const EncodeArgs& a, uint32_t* crc, int nTiles, cudaStream_t s);
cudaError_t launch_record_verify(const uint32_t* computed, const uint32_t* stored, int n, int32_t* status, cudaStream_t s);
// Tile records of rasters with several elements per tile.  elems: device array of nElements descriptors; element e of tile t
// is elems[e].arena[elems[e].offsets[t] .. + elems[e].lens[t]).
struct RecordElement {
  const uint8_t* arena;
  const uint64_t* offsets;
  const uint32_t* lens;
};
// chainLens[t] = sum_e(4 + len_e) - 4: the `lens` argument of launch_record_layout for multi-element records
cudaError_t launch_record_chain_lens(const RecordElement* elems, int nElements, int n, uint32_t* chainLens, cudaStream_t s);
cudaError_t launch_record_pack_multi(const RecordElement* elems, int nElements, const int32_t* tileIndex, int firstTileIndex, int n,
                                     const uint64_t* crcOff, const uint32_t* crcLen, uint8_t* records, int nCtas, cudaStream_t s);
// payloadOff / lens: nElements x n, element-major
cudaError_t launch_record_unpack_multi(const uint8_t* image, uint64_t imageLen, const uint64_t* contentPos, int n, int nElements,
                                       uint64_t* payloadOff, uint32_t* lens, uint64_t* crcOff, uint32_t* crcLen, uint32_t* storedCrc,
                                       int32_t* status, cudaStream_t s);
// a sound record whose CRC differs: status G4_CHECKSUM_MISMATCH, every element's offset and length 0
cudaError_t launch_record_verify_multi(const uint32_t* computed, const uint32_t* stored, int n, int nElements, uint64_t* payloadOff,
                                       uint32_t* lens, int32_t* status, cudaStream_t s);

}  // namespace g4
