// g4_api.cu -- host side of the C ABI declared in include/g4codec.h.
//
// Mirrors the reference's selection layer around the codec kernels:
//   CodecMaster.encodeSingleThread / decode   gvrs/CodecMaster.java:142-203
//   TileElementInt.encode / decode            gvrs/TileElementInt.java:196-219
// (paths under /root/reference/core/src/main/java/org/gridfour/).  No CPU compute path exists here:
// every entry point launches CUDA kernels and fails with G4_ERR_CUDA when that is impossible.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <algorithm>
#include <vector>
#include "g4_kernels.h"

using namespace g4;

namespace {

constexpr int kMaxChunks = 16;  // host-buffer decode pipeline depth (g4_decode_tiles, G4_MEM_HOST)

thread_local std::string tlsError;

int cuda_fail(cudaError_t e, const char* what) {
  tlsError = std::string(what) + ": " + cudaGetErrorString(e);
  return G4_ERR_CUDA;
}
#define CK(call)                                           \
  do {                                                     \
    cudaError_t e_ = (call);                               \
    if (e_ != cudaSuccess) return cuda_fail(e_, #call);    \
  } while (0)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return static_cast<T*>(p); }
};

size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Every entry point runs on its context's device and leaves the caller's current device as it found it (hosts that
// drive several GPUs from one thread -- torch, a JVM -- rely on that).
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != device) err = cudaSetDevice(device);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
#define ENTER(ctx)                                                     \
  DeviceGuard guard_((ctx)->device);                                  \
  if (guard_.err != cudaSuccess) return cuda_fail(guard_.err, "cudaSetDevice")

}  // namespace

struct g4_context {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool ownStream = false;
  int smCount = 148;
  uint64_t launches = 0;
  DevBuf slots[G4_MAX_CODECS];
  DevBuf candLens, candPreds, candStatus;
  DevBuf counters;     // 64 ints: [0..15] encode counters, [16..31] decode counters, [32..47] list counts
  DevBuf scratch;      // per-CTA scratch
  DevBuf lists, src, total;
  DevBuf encScratch;   // per-CTA encoder scratch
  DevBuf region;       // inflate staging (CodecDeflate / CodecFloat decode)
  DevBuf coef;         // LSOP12 decode: 12 float32 coefficients per tile
  DevBuf defer;        // LSOP12 decode: tiles the fast entropy kernel hands to the general one
  DevBuf lsopMeta;     // LSOP12 decode: interior code lengths + text position, kernel H -> kernel T
  DevBuf lsopSide, lsopExc, lsopResid, lsopStage, lsopCks;  // LSOP12 decode, fast path (g4_lsop_fast.cu): side records, exception lists, residual bytes
  DevBuf wide;         // TileElementShort: int32 staging raster around the integer codecs
  DevBuf lsopValueCrc; // LSOP12 encode with G4_LSOP12_VALUE_CHECKSUM: one CRC-32C per tile
  // zlib-stream encode stages (CodecDeflate, CodecFloat, LSOP12 Deflate alternative)
  DevBuf jobLen, jobOff, jobOut, jobTotal, streamIn, streamOut, deflateWork;
  // staged zlib encode (streams <= deflate_staged_max() bytes): sorted positions, bucket ranks, match table, sort tables
  DevBuf stSorted, stRank, stTable, stWork, stCounters;
  // GVRS tile records (g4_records.cu): layout arrays and host-space staging
  DevBuf rcPos, rcOff, rcLen, rcCrc, rcStored, rcTotal, rcData, rcOffsets, rcLens, rcIndex, rcStatus, rcOut;
  DevBuf rcChain, rcDesc;  // multi-element records: per-tile chain lengths, element descriptors (RecordElement)
  std::vector<uint64_t> hostOff;   // jobOff / jobLen mirrored on the host (chunking of the staged encode)
  std::vector<uint32_t> hostLen;
  uint64_t hostTotal = 0;
  int deflateWorkers = 0;   // resident stream-worker threads (0 = default, see g4_context_create)
  uint64_t stagedChunkBytes = 2ull << 30;  // staged zlib encode: input bytes per chunk (scratch = 12x)
  const int64_t* curTileOffset = nullptr;  // tile-list calls: device {offset, pitch} tables of the running call
  const int64_t* curTilePitch = nullptr;
  DevBuf tileRefs;      // device copy of the tile references of a tile-list call
  uint64_t arenaLimit = ~0ull;  // g4_decode_tiles_bounded: bytes addressable behind the arena of the running call
  bool icfOn = false;           // g4_encode_tiles_icf / g4_decode_tiles_icf: the running call's band is G4_ELEM_ICF ...
  g4::IcfMap icf{};             // ... mapped with this descriptor
  // staging used by the host-memory entry points
  DevBuf sGrid, sArena, sOffsets, sLens, sCodec, sPred, sStatus;
  // g4_decode_window: payload locations of the window tiles, absent-tile flags, int32 staging band of unaligned windows
  DevBuf winOff, winLen, winAbsent, winStage;
  // host-buffer decode pipeline: payload H2D / kernels / raster D2H of consecutive chunks overlap
  cudaStream_t copyIn = nullptr, copyOut = nullptr;
  cudaEvent_t evIn[16] = {}, evDone[16] = {}, evStart = nullptr, evOrder = nullptr;
  // optional per-kernel timing (CUDA events on the launching stream): [0]=decode, [1]=encode, by codec kind
  bool timing = false;
  bool asyncDevice = false;  // g4_context_set_async: device batches are enqueued, not awaited
  cudaEvent_t ev[2][G4_CODEC_COUNT + 1][2] = {};
  bool evUsed[2][G4_CODEC_COUNT + 1] = {};
};

namespace {

bool codec_is_float(int id) { return id == G4_CODEC_FLOAT; }

int persistent_ctas(const g4_context* ctx, int nTiles, int perSm) {
  int cap = ctx->smCount * perSm;
  return nTiles < cap ? nTiles : cap;
}

// ---- zlib-stream stages shared by the Deflate-based encoders ---------------------------------------------------------
int ensure_jobs(g4_context* ctx, int nStreams) {
  CK(ctx->jobLen.ensure(size_t(nStreams) * 4));
  CK(ctx->jobOff.ensure(size_t(nStreams) * 8));
  CK(ctx->jobOut.ensure(size_t(nStreams) * 4));
  CK(ctx->jobTotal.ensure(8));
  return G4_OK;
}
// jobLen is filled: offsets, then exact-size staging buffers (one host round trip for the total).
int prepare_streams(g4_context* ctx, int nStreams) {
  CK(launch_stream_offsets(ctx->jobLen.as<uint32_t>(), ctx->jobOff.as<uint64_t>(), nStreams, ctx->jobTotal.as<uint64_t>(), ctx->stream));
  uint64_t total = 0;
  ctx->hostOff.resize(size_t(nStreams) + 1);
  ctx->hostLen.resize(size_t(nStreams));
  CK(cudaMemcpyAsync(&total, ctx->jobTotal.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(ctx->hostOff.data(), ctx->jobOff.p, size_t(nStreams) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(ctx->hostLen.data(), ctx->jobLen.p, size_t(nStreams) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->hostOff[size_t(nStreams)] = total;
  ctx->hostTotal = total;
  CK(ctx->streamIn.ensure(total + 64));
  CK(ctx->streamOut.ensure(total + 112ull * uint64_t(nStreams) + 256));
  ctx->launches++;
  return G4_OK;
}
// zlib streams of the band: the staged kernels (sort / match / emit) take every stream of at most deflate_staged_max()
// bytes, in chunks that bound the per-position scratch (12 bytes per input byte); longer streams go to the general
// one-thread-per-stream kernel.
int run_streams(g4_context* ctx, int nStreams, int capExtra, int level, int* counter) {
  const uint32_t stagedMax = deflate_staged_max();
  int nBig = 0;
  for (int j = 0; j < nStreams; j++) nBig += ctx->hostLen[size_t(j)] > stagedMax;
  if (nBig > 0) {
    int nWorkers = nBig < ctx->deflateWorkers ? nBig : ctx->deflateWorkers;
    nWorkers = (nWorkers + 31) / 32 * 32;
    CK(ctx->deflateWork.ensure(size_t(nWorkers) * deflate_work_bytes()));
    StreamArgs sa{};
    sa.inBuf = ctx->streamIn.as<uint8_t>();
    sa.inOff = ctx->jobOff.as<uint64_t>();
    sa.inLen = ctx->jobLen.as<uint32_t>();
    sa.outBuf = ctx->streamOut.as<uint8_t>();
    sa.outLen = ctx->jobOut.as<uint32_t>();
    sa.nStreams = nStreams;
    sa.capExtra = capExtra;
    sa.level = level;
    sa.work = ctx->deflateWork.p;
    sa.counter = counter;
    sa.bigOnly = 1;
    CK(launch_deflate_streams(sa, nWorkers, ctx->stream));
    ctx->launches++;
  }
  const uint64_t budget = ctx->stagedChunkBytes;
  CK(ctx->stCounters.ensure(4 * sizeof(int)));
  int j0 = 0;
  while (j0 < nStreams) {
    int j1 = j0 + 1;
    while (j1 < nStreams && ctx->hostOff[size_t(j1) + 1] - ctx->hostOff[size_t(j0)] <= budget) j1++;
    const uint64_t base = ctx->hostOff[size_t(j0)];
    const uint64_t span = ctx->hostOff[size_t(j1)] - base;
    const int nChunk = j1 - j0;
    CK(ctx->stSorted.ensure(span * 2 + 64));
    CK(ctx->stRank.ensure(span * 2 + 64));
    CK(ctx->stTable.ensure(span * 8 + 256));
    CK(ctx->stWork.ensure(size_t(nChunk) * deflate_blocks_bytes()));
    CK(cudaMemsetAsync(ctx->stCounters.p, 0, 4 * sizeof(int), ctx->stream));
    StagedArgs st{};
    st.inBuf = ctx->streamIn.as<uint8_t>();
    st.inOff = ctx->jobOff.as<uint64_t>();
    st.inLen = ctx->jobLen.as<uint32_t>();
    st.outBuf = ctx->streamOut.as<uint8_t>();
    st.outLen = ctx->jobOut.as<uint32_t>();
    st.jBegin = j0;
    st.jEnd = j1;
    st.baseOff = base;
    st.sorted = ctx->stSorted.as<uint16_t>();
    st.rank = ctx->stRank.as<uint16_t>();
    st.table = ctx->stTable.as<uint32_t>();
    st.tableQ = ctx->stTable.as<uint32_t>() + (span + 16);
    st.lazy = level >= 9 ? 1 : 0;
    st.maxLen = 0;
    for (int j = j0; j < j1; j++)
      if (ctx->hostLen[size_t(j)] <= stagedMax && ctx->hostLen[size_t(j)] > st.maxLen) st.maxLen = ctx->hostLen[size_t(j)];
    st.blocks = static_cast<DeflateBlocks*>(ctx->stWork.p);
    st.capExtra = capExtra;
    st.level = level;
    st.counters = ctx->stCounters.as<int>();
    CK(launch_deflate_staged(st, ctx->smCount, ctx->stream));
    ctx->launches += st.lazy ? 3 : 4;
    j0 = j1;
  }
  return G4_OK;
}

// Launch one candidate encoder over every tile of the band.  opts: the G4_LSOP12_* option bits of the codec's list entry.
struct KernelTimer;
int launch_encoder_impl(g4_context* ctx, int codecId, int opts, EncodeArgs& a, int nTiles) {
  const int nGrid = persistent_ctas(ctx, nTiles, 8);
  uint32_t* jl = nullptr;
  uint64_t* jo = nullptr;
  uint32_t* jout = nullptr;
  switch (codecId) {
    case G4_CODEC_DEFLATE: {
      const int nStreams = 3 * nTiles;
      int rc = ensure_jobs(ctx, nStreams);
      if (rc != G4_OK) return rc;
      jl = ctx->jobLen.as<uint32_t>(); jo = ctx->jobOff.as<uint64_t>(); jout = ctx->jobOut.as<uint32_t>();
      CK(launch_deflate_m32_size(a, jl, nGrid, ctx->stream));
      if ((rc = prepare_streams(ctx, nStreams)) != G4_OK) return rc;
      CK(launch_deflate_m32_write(a, jl, jo, ctx->streamIn.as<uint8_t>(), nGrid, ctx->stream));
      if ((rc = run_streams(ctx, nStreams, 118, 6, a.counter + 48)) != G4_OK) return rc;
      CK(launch_deflate_pick(a, jl, jo, ctx->streamOut.as<uint8_t>(), jout, nGrid, ctx->stream));
      ctx->launches += 3;
      return G4_OK;
    }
    case G4_CODEC_FLOAT: {
      const int nStreams = 5 * nTiles;
      int rc = ensure_jobs(ctx, nStreams);
      if (rc != G4_OK) return rc;
      jl = ctx->jobLen.as<uint32_t>(); jo = ctx->jobOff.as<uint64_t>(); jout = ctx->jobOut.as<uint32_t>();
      CK(launch_float_plane_size(nTiles, uint32_t(a.band.tile_rows) * uint32_t(a.band.tile_cols), jl, ctx->stream));
      if ((rc = prepare_streams(ctx, nStreams)) != G4_OK) return rc;
      CK(launch_float_plane_write(a, jo, ctx->streamIn.as<uint8_t>(), nGrid, ctx->stream));
      if ((rc = run_streams(ctx, nStreams, 128, 9, a.counter + 48)) != G4_OK) return rc;
      CK(launch_float_pick(a, jo, ctx->streamOut.as<uint8_t>(), jout, nGrid, ctx->stream));
      ctx->launches += 3;
      return G4_OK;
    }
    case G4_CODEC_HUFFMAN: {
      int n = persistent_ctas(ctx, nTiles, 4);
      CK(launch_huffman_encode(a, n, ctx->stream));
      ctx->launches++;
      return G4_OK;
    }
    case G4_CODEC_CANON_HUFFMAN:
    case G4_CODEC_LSOP12: {
      int n = persistent_ctas(ctx, nTiles, 4);
      const size_t stride = 32 * 1024;  // package-merge scratch (g4_canon_enc.cuh)
      CK(ctx->encScratch.ensure(stride * n));
      a.scratch = ctx->encScratch.as<uint8_t>();
      a.scratchStride = stride;
      if (codecId == G4_CODEC_LSOP12 && (opts & G4_LSOP12_VALUE_CHECKSUM)) {  // LsEncoder12.java:128-131
        CK(ctx->lsopValueCrc.ensure(size_t(nTiles) * 4));
        CK(launch_lsop_value_crc(a, ctx->lsopValueCrc.as<uint32_t>(), nTiles, ctx->stream));
        ctx->launches++;
        a.valueCrc = ctx->lsopValueCrc.as<uint32_t>();
      }
      if (codecId == G4_CODEC_CANON_HUFFMAN) CK(launch_canon_encode(a, n, ctx->stream));
      else CK(launch_lsop_encode(a, n, ctx->stream));
      ctx->launches++;
      if (codecId == G4_CODEC_LSOP12 && !(opts & G4_LSOP12_NO_DEFLATE)) {  // LsEncoder12.java:170-218
        const int nStreams = 2 * nTiles;
        int rc = ensure_jobs(ctx, nStreams);
        if (rc != G4_OK) return rc;
        jl = ctx->jobLen.as<uint32_t>(); jo = ctx->jobOff.as<uint64_t>(); jout = ctx->jobOut.as<uint32_t>();
        CK(launch_lsop_m32_size(a, jl, nGrid, ctx->stream));
        if ((rc = prepare_streams(ctx, nStreams)) != G4_OK) return rc;
        CK(launch_lsop_m32_write(a, jl, jo, ctx->streamIn.as<uint8_t>(), nGrid, ctx->stream));
        if ((rc = run_streams(ctx, nStreams, 128, 6, a.counter + 48)) != G4_OK) return rc;
        CK(launch_lsop_pick(a, jl, jo, ctx->streamOut.as<uint8_t>(), jout, nGrid, ctx->stream));
        ctx->launches += 3;
      }
      return G4_OK;
    }
    default:
      tlsError = "codec not implemented on the GPU yet";
      return G4_ERR_UNSUPPORTED;
  }
}

int decoder_ctas(const g4_context* ctx, int nTiles) { return persistent_ctas(ctx, nTiles, 8); }

struct KernelTimer {  // brackets one launch with events when timing is enabled
  g4_context* c;
  int dir, kind;
  KernelTimer(g4_context* ctx, int dir_, int kind_) : c(ctx), dir(dir_), kind(kind_) {
    if (c->timing) {
      if (!c->ev[dir][kind][0]) { cudaEventCreate(&c->ev[dir][kind][0]); cudaEventCreate(&c->ev[dir][kind][1]); }
      cudaEventRecord(c->ev[dir][kind][0], c->stream);
    }
  }
  ~KernelTimer() {
    if (c->timing) { cudaEventRecord(c->ev[dir][kind][1], c->stream); c->evUsed[dir][kind] = true; }
  }
};

int launch_decoder(g4_context* ctx, int codecId, DecodeArgs& a, int nCtas) {
  KernelTimer timer(ctx, 0, codecId);
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  switch (codecId) {
    case G4_CODEC_HUFFMAN: {
      CK(ctx->defer.ensure(size_t(nTiles) * sizeof(int)));
      CK(ctx->lsopStage.ensure(huffman2_spill_bytes(ctx->smCount)));
      CK(ctx->lsopMeta.ensure(huffman2_tree_bytes(nTiles)));
      HuffFusedScratch fused{ctx->lsopStage.as<uint32_t>(), ctx->lsopMeta.as<uint8_t>(), ctx->defer.as<int>(), ctx->counters.as<int>() + 48, ctx->smCount};
      int nLaunch = 0;
      CK(launch_huffman_decode(a, nCtas, ctx->stream, fused, &nLaunch));
      ctx->launches += uint64_t(nLaunch);
      return G4_OK;
    }
    case G4_CODEC_CANON_HUFFMAN:
      CK(launch_canon_decode(a, nCtas, ctx->stream));
      ctx->launches++;
      return G4_OK;
    case G4_CODEC_DEFLATE: {
      const size_t stride = round_up(size_t(a.band.tile_rows) * a.band.tile_cols * 6 + 64, 16);
      CK(ctx->region.ensure(stride * nTiles));
      CK(launch_deflate_decode(a, ctx->region.as<uint8_t>(), stride, nCtas, nTiles, ctx->stream));
      ctx->launches += 2;
      return G4_OK;
    }
    case G4_CODEC_FLOAT: {
      const size_t stride = 5 * round_up(size_t(a.band.tile_rows) * a.band.tile_cols, 16);
      CK(ctx->region.ensure(stride * nTiles));
      CK(launch_float_decode(a, ctx->region.as<uint8_t>(), stride, nCtas, nTiles, ctx->stream));
      ctx->launches += 2;
      return G4_OK;
    }
    case G4_CODEC_LSOP12:
      CK(ctx->coef.ensure(size_t(nTiles) * 12 * sizeof(float)));
      CK(ctx->defer.ensure(size_t(nTiles) * sizeof(int)));
      CK(ctx->lsopMeta.ensure(size_t(nTiles) * lsop_meta_bytes()));
      CK(ctx->lsopCks.ensure(size_t(nTiles) * 8));
      CK(cudaMemsetAsync(ctx->lsopCks.p, 0, size_t(nTiles) * 8, ctx->stream));
      a.lsopCks = ctx->lsopCks.as<uint32_t>();
    {
      int nLaunch = 0;
      LsopFastArgs fast{};
      const bool useFast = lsop_fast_geometry(a.band, a.grid, &fast.g);
      if (useFast) {
        CK(ctx->lsopSide.ensure(lsop_fast_side_bytes(fast.g, nTiles)));
        CK(ctx->lsopExc.ensure(lsop_fast_exc_bytes(nTiles)));
        CK(ctx->lsopResid.ensure(lsop_fast_resid_bytes(fast.g, nTiles)));
        fast.side = ctx->lsopSide.as<int4>();
        fast.exc = ctx->lsopExc.as<uint32_t>();
        fast.resid = ctx->lsopResid.as<uint8_t>();
        if (lsop_fast_stage_bytes(ctx->smCount)) CK(ctx->lsopStage.ensure(lsop_fast_stage_bytes(ctx->smCount)));
        fast.textStage = ctx->lsopStage.as<uint8_t>();
      }
      CK(launch_lsop_decode(a, ctx->coef.as<float>(), ctx->lsopMeta.as<uint8_t>(), ctx->defer.as<int>(), ctx->counters.as<int>() + 56,
                            nCtas, nTiles, ctx->stream, &nLaunch, useFast ? &fast : nullptr, ctx->smCount));
      CK(launch_lsop_value_checksum(a, nTiles, ctx->stream));
      ctx->launches += uint64_t(nLaunch) + 1;
      return G4_OK;
    }
    case G4_CODEC_LSOP08:
      CK(ctx->coef.ensure(size_t(nTiles) * 12 * sizeof(float)));
      CK(launch_lsop08_decode(a, ctx->coef.as<float>(), nCtas, nTiles, ctx->stream));
      ctx->launches += 2;
      return G4_OK;
    default:
      tlsError = "codec not implemented on the GPU yet";
      return G4_ERR_UNSUPPORTED;
  }
}

int launch_encoder(g4_context* ctx, int codecId, int opts, EncodeArgs& a, int nTiles) {
  KernelTimer timer(ctx, 1, codecId);
  return launch_encoder_impl(ctx, codecId, opts, a, nTiles);
}

// A codec-list entry or codec_id argument is a codec id, with the G4_LSOP12_* option bits OR-ed into an LSOP12 entry.
// Splits it into the plain id (what the kernels and every switch on codec ids see) and the bits; G4_ERR_ARG for unknown
// bits or bits on another codec.  Negative entries pass unchanged, for the callers' own checks.
constexpr int32_t kLsop12Options = G4_LSOP12_NO_DEFLATE | G4_LSOP12_VALUE_CHECKSUM;
int split_codec_id(int32_t entry, int32_t* id, int* opts) {
  *id = entry;
  *opts = 0;
  if (entry < 0 || entry <= 0xff) return G4_OK;
  if ((entry & 0xff) != G4_CODEC_LSOP12 || (entry & ~0xff & ~kLsop12Options) != 0) return G4_ERR_ARG;
  *id = G4_CODEC_LSOP12;
  *opts = entry & kLsop12Options;
  return G4_OK;
}
int split_codec_list(const g4_codec_list* in, g4_codec_list* ids, int* opts) {
  if (in->n_codecs < 0 || in->n_codecs > G4_MAX_CODECS) return G4_ERR_ARG;
  *ids = *in;
  for (int k = 0; k < in->n_codecs; k++)
    if (split_codec_id(in->codec_ids[k], &ids->codec_ids[k], &opts[k]) != G4_OK) return G4_ERR_ARG;
  return G4_OK;
}

int check_band(const g4_band_desc* b, bool icf = false) {  // icf: the band of a g4_*_tiles_icf call
  if (!b) return G4_ERR_ARG;
  if (icf ? b->elem_type != G4_ELEM_ICF : b->elem_type != G4_ELEM_I32 && b->elem_type != G4_ELEM_F32 && b->elem_type != G4_ELEM_I16)
    return G4_ERR_ARG;
  if (b->tile_rows < 2 || b->tile_cols < 2) return G4_ERR_UNSUPPORTED;
  if (b->tiles_down < 1 || b->tiles_across < 1) return G4_ERR_ARG;
  if (int64_t(b->tile_rows) * b->tile_cols > (1 << 20)) return G4_ERR_UNSUPPORTED;
  if (b->grid_pitch < int64_t(b->tiles_across) * b->tile_cols) return G4_ERR_ARG;
  if (int64_t(b->tiles_down) * b->tiles_across > (1 << 24)) return G4_ERR_ARG;
  return G4_OK;
}

size_t elem_bytes(const g4_band_desc& b) { return b.elem_type == G4_ELEM_I16 ? 2 : 4; }
// TileElement.standardSizeInBytes (gvrs/TileElement.java:85-93): 4n, or 2n rounded up to a multiple of 4 for shorts
uint32_t standard_size(const g4_band_desc& b) {
  const uint32_t n = uint32_t(b.tile_rows) * uint32_t(b.tile_cols);
  return b.elem_type == G4_ELEM_I16 ? ((2u * n + 3u) & ~3u) : 4u * n;
}

size_t band_samples(const g4_band_desc& b) {
  return size_t(int64_t(b.tiles_down) * b.tile_rows - 1) * size_t(b.grid_pitch) + size_t(b.tiles_across) * b.tile_cols;
}

// Encode with every applicable codec of `codecs`, select, compact.  All pointers are device pointers.
// slotBytes: capacity of each candidate slot.
int encode_device_i32(g4_context* ctx, const g4_codec_list* codecs, const int* opts, const g4_band_desc* band, void* grid, uint8_t* arena,
                      uint64_t arenaCap, uint64_t* offsets, uint32_t* lens, uint8_t* codecOut, uint8_t* predOut, int32_t* status,
                      uint64_t* totalHost, size_t slotBytes, const int16_t* raw16, int64_t raw16Pitch) {
  const int nTiles = band->tiles_down * band->tiles_across;
  const int n = band->tile_rows * band->tile_cols;
  const bool isFloat = band->elem_type == G4_ELEM_F32;
  int cand[G4_MAX_CODECS], nCand = 0;
  for (int k = 0; k < codecs->n_codecs; k++) {
    int id = codecs->codec_ids[k];
    if (id < 0 || id >= G4_CODEC_COUNT) return G4_ERR_ARG;
    if (id == G4_CODEC_LSOP08) continue;  // decode-only legacy codec: its encoder declines every tile
    if (codec_is_float(id) == isFloat) cand[nCand++] = k;
  }
  CK(ctx->candLens.ensure(size_t(nCand + 1) * nTiles * 4));
  CK(ctx->candPreds.ensure(size_t(nCand + 1) * nTiles));
  CK(ctx->candStatus.ensure(size_t(nCand + 1) * nTiles * 4));
  CK(ctx->counters.ensure(64 * sizeof(int)));
  CK(ctx->src.ensure(size_t(nTiles) * 4));
  CK(ctx->total.ensure(8));
  CK(cudaMemsetAsync(ctx->counters.p, 0, 64 * sizeof(int), ctx->stream));
  SelectArgs sel{};
  CompactArgs cmp{};
  for (int c = 0; c < nCand; c++) {
    CK(ctx->slots[c].ensure(size_t(nTiles) * slotBytes));
    EncodeArgs a{};
    a.band = *band;
    a.band.tileOffset = ctx->curTileOffset;
    a.band.tilePitch = ctx->curTilePitch;
    a.grid = grid;
    a.slots = ctx->slots[c].as<uint8_t>();
    a.slotBytes = slotBytes;
    a.lens = ctx->candLens.as<uint32_t>() + size_t(c) * nTiles;
    a.preds = ctx->candPreds.as<uint8_t>() + size_t(c) * nTiles;
    a.status = ctx->candStatus.as<int32_t>() + size_t(c) * nTiles;
    a.counter = ctx->counters.as<int>() + c;
    a.codecIndex = cand[c];
    a.scratch = nullptr;
    a.scratchStride = 0;
    int rc = launch_encoder(ctx, codecs->codec_ids[cand[c]], opts[cand[c]], a, nTiles);
    if (rc != G4_OK) return rc;
    sel.candIndex[c] = cand[c];
    cmp.slots[c] = a.slots;
  }
  sel.nTiles = nTiles;
  sel.nCand = nCand;
  sel.rawLen = raw16 ? ((2u * uint32_t(n) + 3u) & ~3u) : uint32_t(n) * 4u;
  sel.candLens = ctx->candLens.as<uint32_t>();
  sel.candPreds = ctx->candPreds.as<uint8_t>();
  sel.candStatus = ctx->candStatus.as<int32_t>();
  sel.lens = lens;
  sel.codecOut = codecOut;
  sel.predOut = predOut;
  sel.src = ctx->src.as<int>();
  sel.status = status;
  CK(launch_select(sel, ctx->stream));
  CK(launch_offsets(lens, offsets, nTiles, ctx->total.as<uint64_t>(), ctx->stream));
  cmp.band = *band;
  cmp.band.tileOffset = ctx->curTileOffset;
  cmp.band.tilePitch = ctx->curTilePitch;
  cmp.grid = grid;
  cmp.slotBytes = slotBytes;
  cmp.lens = lens;
  cmp.offsets = offsets;
  cmp.src = ctx->src.as<int>();
  cmp.arena = arena;
  cmp.arenaCap = arenaCap;
  cmp.status = status;
  cmp.raw16 = raw16;
  cmp.raw16Pitch = raw16Pitch;
  CK(launch_compact(cmp, nTiles, ctx->stream));
  ctx->launches += 3;
  uint64_t total = 0;
  CK(cudaMemcpyAsync(&total, ctx->total.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (totalHost) *totalHost = total;
  return G4_OK;
}

int decode_device_i32(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, const uint8_t* arena,
                      const uint64_t* offsets, const uint32_t* lens, void* grid, int32_t* status, bool rawShorts) {
  const int nTiles = band->tiles_down * band->tiles_across;
  const int n = band->tile_rows * band->tile_cols;
  const int kinds = G4_CODEC_COUNT + 1;
  CK(ctx->counters.ensure(64 * sizeof(int)));
  CK(ctx->lists.ensure(size_t(kinds) * nTiles * sizeof(int)));
  CK(cudaMemsetAsync(ctx->counters.p, 0, 64 * sizeof(int), ctx->stream));
  ClassifyArgs cl{};
  cl.nTiles = nTiles;
  cl.elemType = band->elem_type;
  cl.rawLen = rawShorts ? ((2u * uint32_t(n) + 3u) & ~3u) : uint32_t(n) * 4u;
  cl.codecs = *codecs;
  cl.arena = arena;
  cl.arenaLen = ctx->arenaLimit;
  cl.offsets = offsets;
  cl.lens = lens;
  cl.lists = ctx->lists.as<int>();
  cl.counts = ctx->counters.as<int>() + 32;
  cl.status = status;
  CK(launch_classify(cl, ctx->stream));
  ctx->launches++;
  const int nCtas = decoder_ctas(ctx, nTiles);
  const size_t stride = round_up(size_t(n) * 6 + 64, 16);
  CK(ctx->scratch.ensure(stride * nCtas));
  bool present[G4_CODEC_COUNT] = {false};
  for (int k = 0; k < codecs->n_codecs; k++) {
    int id = codecs->codec_ids[k];
    if (id < 0 || id >= G4_CODEC_COUNT) return G4_ERR_ARG;
    present[id] = true;
  }
  for (int kind = 0; kind <= G4_CODEC_COUNT; kind++) {
    if (kind < G4_CODEC_COUNT && !present[kind]) continue;
    DecodeArgs a{};
    a.band = *band;
    a.band.tileOffset = ctx->curTileOffset;
    a.band.tilePitch = ctx->curTilePitch;
    a.grid = grid;
    a.arena = arena;
    a.offsets = offsets;
    a.lens = lens;
    a.list = ctx->lists.as<int>() + size_t(kind) * nTiles;
    a.listCount = ctx->counters.as<int>() + 32 + kind;
    a.status = status;
    a.counter = ctx->counters.as<int>() + 16 + kind;
    a.scratch = ctx->scratch.as<uint8_t>();
    a.scratchStride = stride;
    a.rawShorts = rawShorts ? 1 : 0;
    if (kind == G4_CODEC_COUNT) {
      KernelTimer timer(ctx, 0, kind);
      CK(launch_raw_decode(a, nTiles, ctx->stream));
      ctx->launches++;
    } else {
      int rc = launch_decoder(ctx, kind, a, nCtas);
      if (rc != G4_OK) return rc;
    }
  }
  return G4_OK;
}

// TileElementShort around the integer codecs (gvrs/TileElementShort.java:211-248): the 2-byte raster is widened into an
// int32 staging raster (fill value -> INT4_NULL_CODE) before encoding and narrowed after decoding (INT4_NULL_CODE ->
// SHORT_NULL_CODE); raw tiles keep 2 bytes per sample.  All pointers are device pointers.
g4_band_desc widened(const g4_band_desc& b) {
  g4_band_desc w = b;
  w.elem_type = G4_ELEM_I32;
  w.grid_pitch = int64_t(b.tiles_across) * b.tile_cols;
  return w;
}

int encode_device(g4_context* ctx, const g4_codec_list* codecs, const int* opts, const g4_band_desc* band, void* grid, uint8_t* arena,
                  uint64_t arenaCap, uint64_t* offsets, uint32_t* lens, uint8_t* codecOut, uint8_t* predOut, int32_t* status,
                  uint64_t* totalHost, size_t slotBytes) {
  if (band->elem_type == G4_ELEM_ICF) {  // the float band is mapped to codes in the staging raster, which is then encoded
    const g4_band_desc w = widened(*band);
    const int64_t rows = int64_t(band->tiles_down) * band->tile_rows, cols = w.grid_pitch;
    CK(ctx->wide.ensure(size_t(rows) * size_t(cols) * 4));
    CK(launch_icf_map(0, grid, band->grid_pitch, ctx->wide.p, cols, rows, cols, ctx->icf, ctx->stream));
    ctx->launches++;
    return encode_device_i32(ctx, codecs, opts, &w, ctx->wide.p, arena, arenaCap, offsets, lens, codecOut, predOut, status, totalHost, slotBytes,
                             nullptr, 0);
  }
  if (band->elem_type != G4_ELEM_I16)
    return encode_device_i32(ctx, codecs, opts, band, grid, arena, arenaCap, offsets, lens, codecOut, predOut, status, totalHost, slotBytes,
                             nullptr, 0);
  const g4_band_desc w = widened(*band);
  const int64_t rows = int64_t(band->tiles_down) * band->tile_rows, cols = w.grid_pitch;
  CK(ctx->wide.ensure(size_t(rows) * size_t(cols) * 4));
  CK(launch_widen_i16(static_cast<const int16_t*>(grid), band->grid_pitch, ctx->wide.as<int32_t>(), rows, cols, band->fill_value,
                      ctx->stream));
  ctx->launches++;
  return encode_device_i32(ctx, codecs, opts, &w, ctx->wide.p, arena, arenaCap, offsets, lens, codecOut, predOut, status, totalHost, slotBytes,
                           static_cast<const int16_t*>(grid), band->grid_pitch);
}

int decode_device(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, const uint8_t* arena,
                  const uint64_t* offsets, const uint32_t* lens, void* grid, int32_t* status) {
  if (band->elem_type == G4_ELEM_ICF) {  // codes are decoded into the caller's float raster (4 bytes per sample), then mapped in place
    g4_band_desc w = *band;
    w.elem_type = G4_ELEM_I32;
    int rc = decode_device_i32(ctx, codecs, &w, arena, offsets, lens, grid, status, false);
    if (rc != G4_OK) return rc;
    const int64_t rows = int64_t(band->tiles_down) * band->tile_rows, cols = int64_t(band->tiles_across) * band->tile_cols;
    CK(launch_icf_map(1, grid, band->grid_pitch, grid, band->grid_pitch, rows, cols, ctx->icf, ctx->stream));
    ctx->launches++;
    return G4_OK;
  }
  if (band->elem_type != G4_ELEM_I16) return decode_device_i32(ctx, codecs, band, arena, offsets, lens, grid, status, false);
  const g4_band_desc w = widened(*band);
  const int64_t rows = int64_t(band->tiles_down) * band->tile_rows, cols = w.grid_pitch;
  CK(ctx->wide.ensure(size_t(rows) * size_t(cols) * 4));
  int rc = decode_device_i32(ctx, codecs, &w, arena, offsets, lens, ctx->wide.p, status, true);
  if (rc != G4_OK) return rc;
  CK(launch_narrow_i16(ctx->wide.as<int32_t>(), static_cast<int16_t*>(grid), band->grid_pitch, rows, cols, ctx->stream));
  ctx->launches++;
  return G4_OK;
}

int first_bad_status(const std::vector<int32_t>& st) {  // errors before notes (G4_DECLINED, G4_CHECKSUM_MISMATCH)
  int32_t note = G4_OK;
  for (int32_t s : st) {
    if (s < 0) return s;
    if (s != G4_OK && note == G4_OK) note = s;
  }
  return note;
}

}  // namespace

extern "C" {

int g4_abi_version(void) { return G4_ABI_VERSION; }

const char* g4_status_string(int s) {
  switch (s) {
    case G4_OK: return "ok";
    case G4_DECLINED: return "declined (codec returns null for this tile)";
    case G4_ERR_ARG: return "bad argument";
    case G4_ERR_FORMAT: return "malformed packing";
    case G4_ERR_CAPACITY: return "output buffer too small";
    case G4_ERR_CUDA: return "CUDA error";
    case G4_ERR_UNSUPPORTED: return "unsupported";
    default: return "unknown status";
  }
}

const char* g4_last_error(void) { return tlsError.c_str(); }

int g4_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

static const char* kCodecNames[G4_CODEC_COUNT] = {"GvrsHuffman", "GvrsDeflate", "GvrsFloat", "GvrsCanonicalHuffman", "LSOP12", "LSOP08"};

int g4_codec_id_from_name(const char* name) {
  if (!name) return -1;
  for (int i = 0; i < G4_CODEC_COUNT; i++)
    if (std::strcmp(name, kCodecNames[i]) == 0) return i;
  return -1;
}
const char* g4_codec_name(int id) { return (id >= 0 && id < G4_CODEC_COUNT) ? kCodecNames[id] : nullptr; }

int g4_context_create(int device, void* cuda_stream, g4_context** out) {
  if (!out) return G4_ERR_ARG;
  *out = nullptr;
  int nDev = 0;
  cudaError_t e = cudaGetDeviceCount(&nDev);
  if (e != cudaSuccess || nDev == 0) {
    tlsError = "no CUDA device available (the codec kernels have no CPU fallback)";
    return G4_ERR_CUDA;
  }
  if (device < 0 || device >= nDev) return G4_ERR_ARG;
  DeviceGuard guard(device);
  if (guard.err != cudaSuccess) return cuda_fail(guard.err, "cudaSetDevice");
  g4_context* ctx = new g4_context();
  ctx->device = device;
  auto fail = [&](cudaError_t err, const char* what) {
    if (ctx->ownStream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return cuda_fail(err, what);
  };
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(e, "cudaGetDeviceProperties");
  ctx->smCount = prop.multiProcessorCount;
  // resident zlib-stream worker threads: each owns a ~310 KB hash/symbol work area in HBM
  ctx->deflateWorkers = ctx->smCount * 256;
  if (const char* ev = std::getenv("G4_DEFLATE_WORKERS")) { int v = std::atoi(ev); if (v >= 32) ctx->deflateWorkers = v; }
  if (const char* ev = std::getenv("G4_STAGED_CHUNK_MB")) { long v = std::atol(ev); if (v >= 1) ctx->stagedChunkBytes = uint64_t(v) << 20; }
  if (cuda_stream) ctx->stream = static_cast<cudaStream_t>(cuda_stream);
  else {
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "cudaStreamCreateWithFlags");
    ctx->ownStream = true;
  }
  if ((e = cudaEventCreateWithFlags(&ctx->evStart, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreateWithFlags");
  if ((e = cudaEventCreateWithFlags(&ctx->evOrder, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreateWithFlags");
  *out = ctx;
  return G4_OK;
}

// Stream ordering for G4_MEM_DEVICE callers whose buffers are produced / consumed on ANOTHER stream (torch's current
// stream, a JVM's copy stream): work already queued on `other` completes before anything this context launches next
// (before = 1), or everything this context has launched so far completes before `other` continues (before = 0).
int g4_context_order_stream(g4_context* ctx, void* other_stream, int before) {
  if (!ctx) return G4_ERR_ARG;
  cudaStream_t other = static_cast<cudaStream_t>(other_stream);
  if (other == ctx->stream) return G4_OK;
  ENTER(ctx);
  if (before) {
    CK(cudaEventRecord(ctx->evOrder, other));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->evOrder, 0));
  } else {
    CK(cudaEventRecord(ctx->evOrder, ctx->stream));
    CK(cudaStreamWaitEvent(other, ctx->evOrder, 0));
  }
  return G4_OK;
}

void g4_context_destroy(g4_context* ctx) {
  if (!ctx) return;
  DeviceGuard guard(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->copyIn) {
    cudaStreamSynchronize(ctx->copyIn);
    cudaStreamSynchronize(ctx->copyOut);
    cudaStreamDestroy(ctx->copyIn);
    cudaStreamDestroy(ctx->copyOut);
    for (int k = 0; k < kMaxChunks; k++) { cudaEventDestroy(ctx->evIn[k]); cudaEventDestroy(ctx->evDone[k]); }
  }
  if (ctx->evStart) cudaEventDestroy(ctx->evStart);
  if (ctx->evOrder) cudaEventDestroy(ctx->evOrder);
  for (auto& b : ctx->slots) b.release();
  DevBuf* bufs[] = {&ctx->candLens, &ctx->candPreds, &ctx->candStatus, &ctx->counters, &ctx->scratch, &ctx->lists, &ctx->src,
                    &ctx->total, &ctx->coef, &ctx->defer, &ctx->lsopMeta, &ctx->lsopSide, &ctx->lsopExc, &ctx->lsopResid, &ctx->lsopStage, &ctx->tileRefs, &ctx->lsopCks, &ctx->wide, &ctx->encScratch, &ctx->region, &ctx->jobLen, &ctx->jobOff, &ctx->jobOut, &ctx->jobTotal,
                    &ctx->streamIn, &ctx->streamOut, &ctx->deflateWork, &ctx->stSorted, &ctx->stRank, &ctx->stTable,
                    &ctx->stWork, &ctx->stCounters, &ctx->rcPos, &ctx->rcOff, &ctx->rcLen, &ctx->rcCrc, &ctx->rcStored, &ctx->rcTotal,
                    &ctx->rcData, &ctx->rcOffsets, &ctx->rcLens, &ctx->rcIndex, &ctx->rcStatus, &ctx->rcOut, &ctx->rcChain, &ctx->rcDesc, &ctx->sGrid, &ctx->sArena, &ctx->sOffsets, &ctx->sLens, &ctx->sCodec, &ctx->sPred, &ctx->sStatus,
                    &ctx->winOff, &ctx->winLen, &ctx->winAbsent, &ctx->winStage};
  for (DevBuf* b : bufs) b->release();
  if (ctx->ownStream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int g4_context_synchronize(g4_context* ctx) {
  if (!ctx) return G4_ERR_ARG;
  CK(cudaStreamSynchronize(ctx->stream));
  return G4_OK;
}

uint64_t g4_launch_count(const g4_context* ctx) { return ctx ? ctx->launches : 0; }

int g4_context_set_async(g4_context* ctx, int enabled) {
  if (!ctx) return G4_ERR_ARG;
  ctx->asyncDevice = enabled != 0;
  return G4_OK;
}

int g4_context_set_timing(g4_context* ctx, int enabled) {
  if (!ctx) return G4_ERR_ARG;
  ctx->timing = enabled != 0;
  for (auto& d : ctx->evUsed) for (bool& u : d) u = false;
  return G4_OK;
}

int g4_codec_supported(int codec_id, int direction) {
  // direction 0 = decode, 1 = encode.  Grows as codec kernels land; bench.py and the tests ask instead of guessing.
  switch (codec_id) {
    case G4_CODEC_HUFFMAN: return 1;
    case G4_CODEC_DEFLATE: return 1;
    case G4_CODEC_FLOAT: return 1;
    case G4_CODEC_CANON_HUFFMAN: return 1;
    case G4_CODEC_LSOP12: return 1;
    case G4_CODEC_LSOP08: return direction == 0 ? 1 : 0;  // legacy codec: decode only
    default: return 0;
  }
}

double g4_kernel_time_ms(g4_context* ctx, int direction, int codec_kind) {
  if (!ctx || direction < 0 || direction > 1 || codec_kind < 0 || codec_kind > G4_CODEC_COUNT) return -1.0;
  if (!ctx->evUsed[direction][codec_kind]) return -1.0;
  float ms = -1.0f;
  if (cudaEventSynchronize(ctx->ev[direction][codec_kind][1]) != cudaSuccess) return -1.0;
  if (cudaEventElapsedTime(&ms, ctx->ev[direction][codec_kind][0], ctx->ev[direction][codec_kind][1]) != cudaSuccess) return -1.0;
  return double(ms);
}

// ---- GVRS tile records --------------------------------------------------------------------------------------------------
int g4_crc32c(g4_context* ctx, int mem_space, const uint8_t* data, const uint64_t* offsets, const uint32_t* sizes, int n,
              uint32_t* crc_out) {
  if (!ctx || !data || !offsets || !sizes || !crc_out || n < 0) return G4_ERR_ARG;
  if (n == 0) return G4_OK;
  ENTER(ctx);
  if (mem_space == G4_MEM_DEVICE) {
    CK(launch_crc32c(data, offsets, sizes, n, crc_out, 0, ctx->stream));
    ctx->launches++;
    return G4_OK;
  }
  if (mem_space != G4_MEM_HOST) return G4_ERR_ARG;
  uint64_t bytes = 0;
  for (int i = 0; i < n; i++) {
    const uint64_t end = offsets[i] + sizes[i];
    if (end > bytes) bytes = end;
  }
  CK(ctx->rcData.ensure(bytes + 16));
  CK(ctx->rcOff.ensure(size_t(n) * 8));
  CK(ctx->rcLen.ensure(size_t(n) * 4));
  CK(ctx->rcCrc.ensure(size_t(n) * 4));
  CK(cudaMemcpyAsync(ctx->rcData.p, data, bytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->rcOff.p, offsets, size_t(n) * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->rcLen.p, sizes, size_t(n) * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(launch_crc32c(ctx->rcData.as<uint8_t>(), ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(), n, ctx->rcCrc.as<uint32_t>(), 0,
                   ctx->stream));
  ctx->launches++;
  CK(cudaMemcpyAsync(crc_out, ctx->rcCrc.p, size_t(n) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return G4_OK;
}

uint64_t g4_tile_records_bound(int n_tiles, uint64_t payload_bytes) {
  if (n_tiles < 0) return 0;
  return payload_bytes + uint64_t(n_tiles) * 32ull;  // 8 header + 4 index + 4 length + 4 checksum + at most 7 padding
}

int g4_pack_tile_records(g4_context* ctx, int mem_space, const uint8_t* arena, const uint64_t* offsets, const uint32_t* lens,
                         const int32_t* tile_index, int first_tile_index, int n_tiles, int checksum, uint64_t base_pos,
                         uint8_t* records, uint64_t records_cap, uint64_t* content_pos, uint64_t* total_bytes) {
  if (!ctx || !arena || !offsets || !lens || !records || !content_pos || !total_bytes || n_tiles < 0 || (base_pos & 7)) return G4_ERR_ARG;
  if (mem_space != G4_MEM_DEVICE && mem_space != G4_MEM_HOST) return G4_ERR_ARG;
  *total_bytes = 0;
  if (n_tiles == 0) return G4_OK;
  ENTER(ctx);
  const int n = n_tiles;
  const uint8_t* dArena = arena;
  const uint64_t* dOffsets = offsets;
  const uint32_t* dLens = lens;
  const int32_t* dIndex = tile_index;
  uint64_t* dPos = content_pos;
  uint8_t* dRecords = records;
  if (mem_space == G4_MEM_HOST) {
    uint64_t arenaBytes = 0;
    for (int t = 0; t < n; t++) {
      const uint64_t end = offsets[t] + lens[t];
      if (end > arenaBytes) arenaBytes = end;
    }
    CK(ctx->rcData.ensure(arenaBytes + 16));
    CK(ctx->rcOffsets.ensure(size_t(n) * 8));
    CK(ctx->rcLens.ensure(size_t(n) * 4));
    CK(ctx->rcPos.ensure(size_t(n) * 8));
    CK(ctx->rcOut.ensure(records_cap + 16));
    CK(cudaMemcpyAsync(ctx->rcData.p, arena, arenaBytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->rcOffsets.p, offsets, size_t(n) * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->rcLens.p, lens, size_t(n) * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (tile_index) {
      CK(ctx->rcIndex.ensure(size_t(n) * 4));
      CK(cudaMemcpyAsync(ctx->rcIndex.p, tile_index, size_t(n) * 4, cudaMemcpyHostToDevice, ctx->stream));
      dIndex = ctx->rcIndex.as<int32_t>();
    }
    dArena = ctx->rcData.as<uint8_t>();
    dOffsets = ctx->rcOffsets.as<uint64_t>();
    dLens = ctx->rcLens.as<uint32_t>();
    dPos = ctx->rcPos.as<uint64_t>();
    dRecords = ctx->rcOut.as<uint8_t>();
  }
  CK(ctx->rcOff.ensure(size_t(n) * 8));
  CK(ctx->rcLen.ensure(size_t(n) * 4));
  CK(ctx->rcTotal.ensure(8));
  CK(launch_record_layout(dLens, n, base_pos, dPos, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(), ctx->rcTotal.as<uint64_t>(),
                          ctx->stream));
  uint64_t total = 0;
  CK(cudaMemcpyAsync(&total, ctx->rcTotal.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *total_bytes = total;
  if (total > records_cap) return G4_ERR_CAPACITY;
  CK(launch_record_pack(dArena, dOffsets, dLens, dIndex, first_tile_index, n, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(), dRecords,
                        persistent_ctas(ctx, n, 8), ctx->stream));
  ctx->launches += 2;
  if (checksum) {
    CK(launch_crc32c(dRecords, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(), n, nullptr, 1, ctx->stream));
    ctx->launches++;
  }
  if (mem_space == G4_MEM_HOST) {
    CK(cudaMemcpyAsync(records, dRecords, total, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(content_pos, dPos, size_t(n) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return G4_OK;
}

int g4_unpack_tile_records(g4_context* ctx, int mem_space, const uint8_t* image, uint64_t image_len, const uint64_t* content_pos,
                           int n_tiles, int checksum, uint64_t* payload_offsets, uint32_t* lens, int32_t* status) {
  if (!ctx || !image || !content_pos || !payload_offsets || !lens || !status || n_tiles < 0) return G4_ERR_ARG;
  if (mem_space != G4_MEM_DEVICE && mem_space != G4_MEM_HOST) return G4_ERR_ARG;
  if (n_tiles == 0) return G4_OK;
  ENTER(ctx);
  const int n = n_tiles;
  const uint8_t* dImage = image;
  const uint64_t* dPos = content_pos;
  uint64_t* dPay = payload_offsets;
  uint32_t* dLens = lens;
  int32_t* dStatus = status;
  if (mem_space == G4_MEM_HOST) {
    CK(ctx->rcData.ensure(image_len + 16));
    CK(ctx->rcPos.ensure(size_t(n) * 8));
    CK(ctx->rcOffsets.ensure(size_t(n) * 8));
    CK(ctx->rcLens.ensure(size_t(n) * 4));
    CK(ctx->rcStatus.ensure(size_t(n) * 4));
    CK(cudaMemcpyAsync(ctx->rcData.p, image, image_len, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->rcPos.p, content_pos, size_t(n) * 8, cudaMemcpyHostToDevice, ctx->stream));
    dImage = ctx->rcData.as<uint8_t>();
    dPos = ctx->rcPos.as<uint64_t>();
    dPay = ctx->rcOffsets.as<uint64_t>();
    dLens = ctx->rcLens.as<uint32_t>();
    dStatus = ctx->rcStatus.as<int32_t>();
  }
  if (reinterpret_cast<uintptr_t>(dImage) & 7) return G4_ERR_ARG;
  CK(ctx->rcOff.ensure(size_t(n) * 8));
  CK(ctx->rcLen.ensure(size_t(n) * 4));
  CK(ctx->rcCrc.ensure(size_t(n) * 4));
  CK(ctx->rcStored.ensure(size_t(n) * 4));
  CK(launch_record_unpack(dImage, image_len, dPos, n, dPay, dLens, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(),
                          ctx->rcStored.as<uint32_t>(), dStatus, ctx->stream));
  ctx->launches++;
  if (checksum) {
    CK(launch_crc32c(dImage, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(), n, ctx->rcCrc.as<uint32_t>(), 0, ctx->stream));
    CK(launch_record_verify(ctx->rcCrc.as<uint32_t>(), ctx->rcStored.as<uint32_t>(), n, dStatus, ctx->stream));
    ctx->launches += 2;
  }
  if (mem_space == G4_MEM_HOST) {
    CK(cudaMemcpyAsync(payload_offsets, dPay, size_t(n) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(lens, dLens, size_t(n) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(status, dStatus, size_t(n) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return G4_OK;
}

uint64_t g4_tile_records_bound_multi(int n_tiles, int n_elements, uint64_t payload_bytes) {
  if (n_tiles < 0 || n_elements < 1 || n_elements > G4_MAX_ELEMENTS) return 0;
  // 8 header + 4 index + 4 length per element + 4 checksum + at most 7 padding
  return payload_bytes + uint64_t(n_tiles) * (23ull + 4ull * uint64_t(n_elements));
}

int g4_pack_tile_records_multi(g4_context* ctx, int mem_space, int n_elements, const uint8_t* const* arenas,
                               const uint64_t* const* offsets, const uint32_t* const* lens, const int32_t* tile_index,
                               int first_tile_index, int n_tiles, int checksum, uint64_t base_pos, uint8_t* records,
                               uint64_t records_cap, uint64_t* content_pos, uint64_t* total_bytes) {
  if (!ctx || !arenas || !offsets || !lens || !records || !content_pos || !total_bytes || n_tiles < 0 || (base_pos & 7)) return G4_ERR_ARG;
  if (n_elements < 1 || n_elements > G4_MAX_ELEMENTS) return G4_ERR_UNSUPPORTED;
  if (mem_space != G4_MEM_DEVICE && mem_space != G4_MEM_HOST) return G4_ERR_ARG;
  for (int e = 0; e < n_elements; e++)
    if (!arenas[e] || !offsets[e] || !lens[e]) return G4_ERR_ARG;
  *total_bytes = 0;
  if (n_tiles == 0) return G4_OK;
  ENTER(ctx);
  const int n = n_tiles, E = n_elements;
  std::vector<RecordElement> desc(static_cast<size_t>(E));
  const int32_t* dIndex = tile_index;
  uint64_t* dPos = content_pos;
  uint8_t* dRecords = records;
  if (mem_space == G4_MEM_HOST) {
    // every element's used arena range, back to back (16-byte aligned) in rcData; offsets and lengths element-major
    std::vector<uint64_t> base(size_t(E) + 1, 0), used(size_t(E), 0);
    for (int e = 0; e < E; e++) {
      for (int t = 0; t < n; t++) {
        const uint64_t end = offsets[e][t] + lens[e][t];
        if (end > used[size_t(e)]) used[size_t(e)] = end;
      }
      base[size_t(e) + 1] = round_up(base[size_t(e)] + used[size_t(e)], 16);
    }
    CK(ctx->rcData.ensure(base[size_t(E)] + 16));
    CK(ctx->rcOffsets.ensure(size_t(E) * n * 8));
    CK(ctx->rcLens.ensure(size_t(E) * n * 4));
    CK(ctx->rcPos.ensure(size_t(n) * 8));
    CK(ctx->rcOut.ensure(records_cap + 16));
    for (int e = 0; e < E; e++) {
      uint8_t* a = ctx->rcData.as<uint8_t>() + base[size_t(e)];
      uint64_t* o = ctx->rcOffsets.as<uint64_t>() + size_t(e) * n;
      uint32_t* l = ctx->rcLens.as<uint32_t>() + size_t(e) * n;
      if (used[size_t(e)]) CK(cudaMemcpyAsync(a, arenas[e], used[size_t(e)], cudaMemcpyHostToDevice, ctx->stream));
      CK(cudaMemcpyAsync(o, offsets[e], size_t(n) * 8, cudaMemcpyHostToDevice, ctx->stream));
      CK(cudaMemcpyAsync(l, lens[e], size_t(n) * 4, cudaMemcpyHostToDevice, ctx->stream));
      desc[size_t(e)] = RecordElement{a, o, l};
    }
    if (tile_index) {
      CK(ctx->rcIndex.ensure(size_t(n) * 4));
      CK(cudaMemcpyAsync(ctx->rcIndex.p, tile_index, size_t(n) * 4, cudaMemcpyHostToDevice, ctx->stream));
      dIndex = ctx->rcIndex.as<int32_t>();
    }
    dPos = ctx->rcPos.as<uint64_t>();
    dRecords = ctx->rcOut.as<uint8_t>();
  } else {
    for (int e = 0; e < E; e++) desc[size_t(e)] = RecordElement{arenas[e], offsets[e], lens[e]};
  }
  CK(ctx->rcDesc.ensure(size_t(E) * sizeof(RecordElement)));
  CK(cudaMemcpyAsync(ctx->rcDesc.p, desc.data(), size_t(E) * sizeof(RecordElement), cudaMemcpyHostToDevice, ctx->stream));
  const RecordElement* dDesc = ctx->rcDesc.as<RecordElement>();
  CK(ctx->rcChain.ensure(size_t(n) * 4));
  CK(ctx->rcOff.ensure(size_t(n) * 8));
  CK(ctx->rcLen.ensure(size_t(n) * 4));
  CK(ctx->rcTotal.ensure(8));
  CK(launch_record_chain_lens(dDesc, E, n, ctx->rcChain.as<uint32_t>(), ctx->stream));
  CK(launch_record_layout(ctx->rcChain.as<uint32_t>(), n, base_pos, dPos, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(),
                          ctx->rcTotal.as<uint64_t>(), ctx->stream));
  uint64_t total = 0;
  CK(cudaMemcpyAsync(&total, ctx->rcTotal.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));  // (also the end of `desc`'s copy)
  ctx->launches += 2;
  *total_bytes = total;
  if (total > records_cap) return G4_ERR_CAPACITY;
  CK(launch_record_pack_multi(dDesc, E, dIndex, first_tile_index, n, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(), dRecords,
                              persistent_ctas(ctx, n, 8), ctx->stream));
  ctx->launches++;
  if (checksum) {
    CK(launch_crc32c(dRecords, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(), n, nullptr, 1, ctx->stream));
    ctx->launches++;
  }
  if (mem_space == G4_MEM_HOST) {
    CK(cudaMemcpyAsync(records, dRecords, total, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(content_pos, dPos, size_t(n) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return G4_OK;
}

int g4_unpack_tile_records_multi(g4_context* ctx, int mem_space, int n_elements, const uint8_t* image, uint64_t image_len,
                                 const uint64_t* content_pos, int n_tiles, int checksum, uint64_t* payload_offsets,
                                 uint32_t* lens, int32_t* status) {
  if (!ctx || !image || !content_pos || !payload_offsets || !lens || !status || n_tiles < 0) return G4_ERR_ARG;
  if (n_elements < 1 || n_elements > G4_MAX_ELEMENTS) return G4_ERR_UNSUPPORTED;
  if (mem_space != G4_MEM_DEVICE && mem_space != G4_MEM_HOST) return G4_ERR_ARG;
  if (n_tiles == 0) return G4_OK;
  ENTER(ctx);
  const int n = n_tiles, E = n_elements;
  const uint8_t* dImage = image;
  const uint64_t* dPos = content_pos;
  uint64_t* dPay = payload_offsets;
  uint32_t* dLens = lens;
  int32_t* dStatus = status;
  if (mem_space == G4_MEM_HOST) {
    CK(ctx->rcData.ensure(image_len + 16));
    CK(ctx->rcPos.ensure(size_t(n) * 8));
    CK(ctx->rcOffsets.ensure(size_t(E) * n * 8));
    CK(ctx->rcLens.ensure(size_t(E) * n * 4));
    CK(ctx->rcStatus.ensure(size_t(n) * 4));
    CK(cudaMemcpyAsync(ctx->rcData.p, image, image_len, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->rcPos.p, content_pos, size_t(n) * 8, cudaMemcpyHostToDevice, ctx->stream));
    dImage = ctx->rcData.as<uint8_t>();
    dPos = ctx->rcPos.as<uint64_t>();
    dPay = ctx->rcOffsets.as<uint64_t>();
    dLens = ctx->rcLens.as<uint32_t>();
    dStatus = ctx->rcStatus.as<int32_t>();
  }
  if (reinterpret_cast<uintptr_t>(dImage) & 7) return G4_ERR_ARG;
  CK(ctx->rcOff.ensure(size_t(n) * 8));
  CK(ctx->rcLen.ensure(size_t(n) * 4));
  CK(ctx->rcCrc.ensure(size_t(n) * 4));
  CK(ctx->rcStored.ensure(size_t(n) * 4));
  CK(launch_record_unpack_multi(dImage, image_len, dPos, n, E, dPay, dLens, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(),
                                ctx->rcStored.as<uint32_t>(), dStatus, ctx->stream));
  ctx->launches++;
  if (checksum) {
    CK(launch_crc32c(dImage, ctx->rcOff.as<uint64_t>(), ctx->rcLen.as<uint32_t>(), n, ctx->rcCrc.as<uint32_t>(), 0, ctx->stream));
    CK(launch_record_verify_multi(ctx->rcCrc.as<uint32_t>(), ctx->rcStored.as<uint32_t>(), n, E, dPay, dLens, dStatus, ctx->stream));
    ctx->launches += 2;
  }
  if (mem_space == G4_MEM_HOST) {
    CK(cudaMemcpyAsync(payload_offsets, dPay, size_t(E) * n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(lens, dLens, size_t(E) * n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(status, dStatus, size_t(n) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return G4_OK;
}

uint64_t g4_encode_arena_bound(const g4_band_desc* b) {
  if (!b) return 0;
  uint64_t n = uint64_t(b->tile_rows) * b->tile_cols;
  return uint64_t(b->tiles_down) * b->tiles_across * ((n * 4 + 7) & ~7ull);
}

int g4_fill_terrain(g4_context* ctx, int elem_type, uint64_t seed, int64_t row0, int64_t col0, int64_t n_rows, int64_t n_cols,
                    void* device_out) {
  if (!ctx || !device_out || n_rows < 1 || n_cols < 1) return G4_ERR_ARG;
  ENTER(ctx);
  CK(launch_fill_terrain(elem_type, seed, row0, col0, n_rows, n_cols, device_out, ctx->stream));
  ctx->launches++;
  return G4_OK;
}

// Tile-list calls: `refs` (host array, one {offset, pitch} per tile, in samples relative to `grid`) replaces the tile grid
// of the band, which is then a list of band->tiles_across tiles.  Device rasters are addressed in place through the
// per-tile tables of BandEx; host rasters are staged tile under tile by 2-D copies (no host gather).
static int upload_tile_refs(g4_context* ctx, const g4_tile_ref* refs, int nTiles) {
  std::vector<int64_t> h(size_t(nTiles) * 2);
  for (int t = 0; t < nTiles; t++) { h[size_t(t)] = refs[t].offset; h[size_t(nTiles) + t] = refs[t].pitch; }
  CK(ctx->tileRefs.ensure(h.size() * 8));
  CK(cudaMemcpyAsync(ctx->tileRefs.p, h.data(), h.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));  // h goes out of scope
  ctx->curTileOffset = ctx->tileRefs.as<int64_t>();
  ctx->curTilePitch = ctx->tileRefs.as<int64_t>() + nTiles;
  return G4_OK;
}
struct TileRefScope {  // the tables are valid for one call only
  g4_context* c;
  ~TileRefScope() { c->curTileOffset = nullptr; c->curTilePitch = nullptr; }
};

static int encode_tiles_impl(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space, const void* grid,
                             const g4_tile_ref* refs, uint8_t* arena, uint64_t arena_cap, uint64_t* offsets, uint32_t* lens,
                             uint8_t* codec_out, uint8_t* predictor_out, int32_t* status, uint64_t* total_bytes) {
  if (!ctx || !codecs || !grid || !arena || !offsets || !lens || !codec_out || !predictor_out || !status) return G4_ERR_ARG;
  int rc = check_band(band, ctx->icfOn);
  if (rc != G4_OK) return rc;
  g4_codec_list ids;
  int opts[G4_MAX_CODECS];
  if (split_codec_list(codecs, &ids, opts) != G4_OK) return G4_ERR_ARG;
  codecs = &ids;
  ENTER(ctx);
  const int nTiles = band->tiles_down * band->tiles_across;
  const size_t n = size_t(band->tile_rows) * band->tile_cols;
  const size_t slotBytes = round_up(n * 4 + 64, 16);
  const size_t eb = elem_bytes(*band);
  std::vector<int32_t> st(nTiles);
  uint64_t total = 0;
  TileRefScope scope{ctx};
  if (mem_space == G4_MEM_DEVICE) {
    if (refs && (rc = upload_tile_refs(ctx, refs, nTiles)) != G4_OK) return rc;
    rc = encode_device(ctx, codecs, opts, band, const_cast<void*>(grid), arena, arena_cap, offsets, lens, codec_out, predictor_out,
                       status, &total, slotBytes);
    if (rc != G4_OK) return rc;
    CK(cudaMemcpyAsync(st.data(), status, size_t(nTiles) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  } else if (mem_space == G4_MEM_HOST) {
    g4_band_desc staged = *band;
    if (refs) {  // the tiles go tile under tile into one staging raster of pitch tile_cols
      staged.tiles_down = nTiles;
      staged.tiles_across = 1;
      staged.grid_pitch = band->tile_cols;
    }
    const size_t gridBytes = band_samples(staged) * eb;
    const uint64_t bound = g4_encode_arena_bound(band);
    CK(ctx->sGrid.ensure(gridBytes));
    CK(ctx->sArena.ensure(bound + 16));
    CK(ctx->sOffsets.ensure(size_t(nTiles) * 8));
    CK(ctx->sLens.ensure(size_t(nTiles) * 4));
    CK(ctx->sCodec.ensure(nTiles));
    CK(ctx->sPred.ensure(nTiles));
    CK(ctx->sStatus.ensure(size_t(nTiles) * 4));
    if (refs) {
      for (int t = 0; t < nTiles; t++)
        CK(cudaMemcpy2DAsync(ctx->sGrid.as<uint8_t>() + size_t(t) * n * eb, size_t(band->tile_cols) * eb,
                             static_cast<const uint8_t*>(grid) + refs[t].offset * int64_t(eb), size_t(refs[t].pitch) * eb,
                             size_t(band->tile_cols) * eb, size_t(band->tile_rows), cudaMemcpyHostToDevice, ctx->stream));
    } else CK(cudaMemcpyAsync(ctx->sGrid.p, grid, gridBytes, cudaMemcpyHostToDevice, ctx->stream));
    band = &staged;
    rc = encode_device(ctx, codecs, opts, band, ctx->sGrid.p, ctx->sArena.as<uint8_t>(), bound, ctx->sOffsets.as<uint64_t>(),
                       ctx->sLens.as<uint32_t>(), ctx->sCodec.as<uint8_t>(), ctx->sPred.as<uint8_t>(), ctx->sStatus.as<int32_t>(),
                       &total, slotBytes);
    if (rc != G4_OK) return rc;
    if (total > arena_cap) {
      if (total_bytes) *total_bytes = total;
      return G4_ERR_CAPACITY;
    }
    CK(cudaMemcpyAsync(arena, ctx->sArena.p, total, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(offsets, ctx->sOffsets.p, size_t(nTiles) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(lens, ctx->sLens.p, size_t(nTiles) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(codec_out, ctx->sCodec.p, nTiles, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(predictor_out, ctx->sPred.p, nTiles, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(status, ctx->sStatus.p, size_t(nTiles) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    std::memcpy(st.data(), status, size_t(nTiles) * 4);
  } else {
    return G4_ERR_ARG;
  }
  if (total_bytes) *total_bytes = total;
  return first_bad_status(st);
}

int g4_encode_tiles(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space, const void* grid,
                    uint8_t* arena, uint64_t arena_cap, uint64_t* offsets, uint32_t* lens, uint8_t* codec_out,
                    uint8_t* predictor_out, int32_t* status, uint64_t* total_bytes) {
  return encode_tiles_impl(ctx, codecs, band, mem_space, grid, nullptr, arena, arena_cap, offsets, lens, codec_out, predictor_out, status,
                           total_bytes);
}

// The band a tile list runs as: one row of n tiles.  grid_pitch only carries the ALIGNMENT the kernels may rely on (the
// vectorised LSOP12 paths test it modulo 4 and 8); the per-tile tables give the real geometry.
static int tile_list_band(int elem_type, int tile_rows, int tile_cols, int n_tiles, const g4_tile_ref* refs, g4_band_desc* out) {
  if (!refs || n_tiles < 1 || (elem_type != G4_ELEM_I32 && elem_type != G4_ELEM_F32)) return elem_type == G4_ELEM_I16 ? G4_ERR_UNSUPPORTED : G4_ERR_ARG;
  int align = 8;
  for (int t = 0; t < n_tiles; t++) {
    if (refs[t].pitch < tile_cols || refs[t].offset < 0) return G4_ERR_ARG;
    while (align > 1 && ((refs[t].offset % align) != 0 || (refs[t].pitch % align) != 0)) align >>= 1;
  }
  int64_t rep = ((int64_t(n_tiles) * tile_cols + 7) / 8) * 8;
  if (align == 4) rep += 4;
  else if (align < 4) rep += 1;
  *out = g4_band_desc{elem_type, tile_rows, tile_cols, 1, n_tiles, rep, 0, 0};
  return G4_OK;
}

int g4_encode_tile_list(g4_context* ctx, const g4_codec_list* codecs, int elem_type, int tile_rows, int tile_cols, int n_tiles,
                        int mem_space, const void* base, const g4_tile_ref* tiles, uint8_t* arena, uint64_t arena_cap, uint64_t* offsets,
                        uint32_t* lens, uint8_t* codec_out, uint8_t* predictor_out, int32_t* status, uint64_t* total_bytes) {
  g4_band_desc band;
  const int rc = tile_list_band(elem_type, tile_rows, tile_cols, n_tiles, tiles, &band);
  if (rc != G4_OK) return rc;
  return encode_tiles_impl(ctx, codecs, &band, mem_space, base, tiles, arena, arena_cap, offsets, lens, codec_out, predictor_out, status,
                           total_bytes);
}

static int decode_tiles_impl(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space, const uint8_t* arena,
                             const uint64_t* offsets, const uint32_t* lens, void* grid, const g4_tile_ref* refs, int32_t* status) {
  if (!ctx || !codecs || !grid || !arena || !offsets || !lens || !status) return G4_ERR_ARG;
  int rc = check_band(band, ctx->icfOn);
  if (rc != G4_OK) return rc;
  g4_codec_list ids;  // decode ignores the option bits: they describe how to encode, the packings say the rest
  int opts[G4_MAX_CODECS];
  if (split_codec_list(codecs, &ids, opts) != G4_OK) return G4_ERR_ARG;
  codecs = &ids;
  ENTER(ctx);
  const int nTiles = band->tiles_down * band->tiles_across;
  std::vector<int32_t> st(nTiles);
  TileRefScope scope{ctx};
  if (mem_space == G4_MEM_DEVICE) {
    if (refs && (rc = upload_tile_refs(ctx, refs, nTiles)) != G4_OK) return rc;
    rc = decode_device(ctx, codecs, band, arena, offsets, lens, grid, status);
    if (rc != G4_OK) return rc;
    if (ctx->asyncDevice && !refs) return G4_OK;  // enqueued; status[] is read by the caller after g4_context_synchronize
    CK(cudaMemcpyAsync(st.data(), status, size_t(nTiles) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  } else if (mem_space == G4_MEM_HOST) {
    // a directory entry that leaves the caller's arena (g4_decode_tiles_bounded) or is longer than the raw tile is never
    // staged: it reaches the device as an empty payload, which classify_kernel reports as G4_ERR_FORMAT for that tile
    std::vector<uint64_t> offSafe;
    std::vector<uint32_t> lenSafe;
    const uint32_t rawLen = standard_size(*band);
    for (int t = 0; t < nTiles; t++) {
      const bool bad = lens[t] > rawLen || (ctx->arenaLimit != ~0ull && (offsets[t] > ctx->arenaLimit || lens[t] > ctx->arenaLimit - offsets[t]));
      if (bad && offSafe.empty()) {
        offSafe.assign(offsets, offsets + nTiles);
        lenSafe.assign(lens, lens + nTiles);
      }
      if (bad) { offSafe[size_t(t)] = 0; lenSafe[size_t(t)] = 0; }
    }
    if (!offSafe.empty()) { offsets = offSafe.data(); lens = lenSafe.data(); }
    uint64_t arenaBytes = 0;
    for (int t = 0; t < nTiles; t++) {
      uint64_t end = offsets[t] + lens[t];
      if (end > arenaBytes) arenaBytes = end;
    }
    g4_band_desc staged = *band;
    if (refs) {  // decode tile under tile into one staging raster of pitch tile_cols, then one 2-D copy per tile
      staged.tiles_down = nTiles;
      staged.tiles_across = 1;
      staged.grid_pitch = band->tile_cols;
      band = &staged;
    }
    const size_t gridBytes = band_samples(*band) * elem_bytes(*band);
    const size_t rowBytes = size_t(band->grid_pitch) * elem_bytes(*band);
    const size_t bandRowBytes = size_t(band->tiles_across) * band->tile_cols * elem_bytes(*band);
    const size_t bandRows = size_t(band->tiles_down) * band->tile_rows;
    const bool pitched = rowBytes != bandRowBytes;
    CK(ctx->sGrid.ensure(gridBytes));
    CK(ctx->sArena.ensure(arenaBytes + 16));
    CK(ctx->sOffsets.ensure(size_t(nTiles) * 8));
    CK(ctx->sLens.ensure(size_t(nTiles) * 4));
    CK(ctx->sStatus.ensure(size_t(nTiles) * 4));
    CK(cudaMemcpyAsync(ctx->sOffsets.p, offsets, size_t(nTiles) * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->sLens.p, lens, size_t(nTiles) * 4, cudaMemcpyHostToDevice, ctx->stream));
    // The decoded raster (4 B/sample) crossing PCIe dominates this call, so the band is cut into chunks of whole tile
    // rows and pipelined over three streams: payload H2D of chunk k+1, kernels of chunk k and raster D2H of chunk k-1
    // overlap.  Needs payloads in ascending tile order (what g4_encode_tiles produces); otherwise one chunk.
    bool ascending = true;
    for (int t = 1; t < nTiles && ascending; t++) ascending = offsets[t] >= offsets[t - 1] + lens[t - 1];
    int nChunks = ascending ? (band->tiles_down < kMaxChunks ? band->tiles_down : kMaxChunks) : 1;
    if (gridBytes < (size_t(32) << 20) || refs) nChunks = 1;  // small bands: the fixed cost per chunk is not worth it
    if (nChunks > 1 && !ctx->copyIn) {
      CK(cudaStreamCreateWithFlags(&ctx->copyIn, cudaStreamNonBlocking));
      CK(cudaStreamCreateWithFlags(&ctx->copyOut, cudaStreamNonBlocking));
      for (int k = 0; k < kMaxChunks; k++) {
        CK(cudaEventCreateWithFlags(&ctx->evIn[k], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->evDone[k], cudaEventDisableTiming));
      }
    }
    if (nChunks == 1) {
      CK(cudaMemcpyAsync(ctx->sArena.p, arena, arenaBytes, cudaMemcpyHostToDevice, ctx->stream));
      rc = decode_device(ctx, codecs, band, ctx->sArena.as<uint8_t>(), ctx->sOffsets.as<uint64_t>(), ctx->sLens.as<uint32_t>(),
                         ctx->sGrid.p, ctx->sStatus.as<int32_t>());
      if (rc != G4_OK) return rc;
      if (refs) {
        const size_t eb = elem_bytes(*band), tileBytes = size_t(band->tile_rows) * band->tile_cols * eb;
        for (int t = 0; t < nTiles; t++)
          CK(cudaMemcpy2DAsync(static_cast<uint8_t*>(grid) + refs[t].offset * int64_t(eb), size_t(refs[t].pitch) * eb,
                               ctx->sGrid.as<uint8_t>() + size_t(t) * tileBytes, size_t(band->tile_cols) * eb, size_t(band->tile_cols) * eb,
                               size_t(band->tile_rows), cudaMemcpyDeviceToHost, ctx->stream));
      } else if (pitched)  // a band inside a wider host raster: only the band's columns go back
        CK(cudaMemcpy2DAsync(grid, rowBytes, ctx->sGrid.p, rowBytes, bandRowBytes, bandRows, cudaMemcpyDeviceToHost, ctx->stream));
      else
        CK(cudaMemcpyAsync(grid, ctx->sGrid.p, gridBytes, cudaMemcpyDeviceToHost, ctx->stream));
    } else {
      CK(cudaEventRecord(ctx->evStart, ctx->stream));
      CK(cudaStreamWaitEvent(ctx->copyIn, ctx->evStart, 0));   // the staging buffers may still be in use by an earlier call
      CK(cudaStreamWaitEvent(ctx->copyOut, ctx->evStart, 0));
      for (int k = 0; k < nChunks; k++) {
        const int r0 = int(int64_t(band->tiles_down) * k / nChunks), r1 = int(int64_t(band->tiles_down) * (k + 1) / nChunks);
        const int t0 = r0 * band->tiles_across, t1 = r1 * band->tiles_across;
        const uint64_t lo = offsets[t0], hi = offsets[t1 - 1] + lens[t1 - 1];
        CK(cudaMemcpyAsync(ctx->sArena.as<uint8_t>() + lo, arena + lo, hi - lo, cudaMemcpyHostToDevice, ctx->copyIn));
        CK(cudaEventRecord(ctx->evIn[k], ctx->copyIn));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->evIn[k], 0));
        g4_band_desc sub = *band;
        sub.tiles_down = r1 - r0;
        uint8_t* gdev = ctx->sGrid.as<uint8_t>() + size_t(r0) * band->tile_rows * rowBytes;
        rc = decode_device(ctx, codecs, &sub, ctx->sArena.as<uint8_t>(), ctx->sOffsets.as<uint64_t>() + t0, ctx->sLens.as<uint32_t>() + t0,
                           gdev, ctx->sStatus.as<int32_t>() + t0);
        if (rc != G4_OK) return rc;
        CK(cudaEventRecord(ctx->evDone[k], ctx->stream));
        CK(cudaStreamWaitEvent(ctx->copyOut, ctx->evDone[k], 0));
        const size_t rows = size_t(r1 - r0) * band->tile_rows;
        const size_t bytes = k == nChunks - 1 ? gridBytes - size_t(r0) * band->tile_rows * rowBytes : rows * rowBytes;
        uint8_t* ghost = static_cast<uint8_t*>(grid) + size_t(r0) * band->tile_rows * rowBytes;
        if (pitched) CK(cudaMemcpy2DAsync(ghost, rowBytes, gdev, rowBytes, bandRowBytes, rows, cudaMemcpyDeviceToHost, ctx->copyOut));
        else CK(cudaMemcpyAsync(ghost, gdev, bytes, cudaMemcpyDeviceToHost, ctx->copyOut));
      }
      CK(cudaEventRecord(ctx->evIn[0], ctx->copyOut));
      CK(cudaStreamWaitEvent(ctx->stream, ctx->evIn[0], 0));  // the call's stream completes only after the last D2H
    }
    CK(cudaMemcpyAsync(status, ctx->sStatus.p, size_t(nTiles) * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    std::memcpy(st.data(), status, size_t(nTiles) * 4);
  } else {
    return G4_ERR_ARG;
  }
  return first_bad_status(st);
}

int g4_decode_tiles(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space, const uint8_t* arena,
                    const uint64_t* offsets, const uint32_t* lens, void* grid, int32_t* status) {
  return decode_tiles_impl(ctx, codecs, band, mem_space, arena, offsets, lens, grid, nullptr, status);
}

int g4_decode_tile_list(g4_context* ctx, const g4_codec_list* codecs, int elem_type, int tile_rows, int tile_cols, int n_tiles,
                        int mem_space, const uint8_t* arena, uint64_t arena_len, const uint64_t* offsets, const uint32_t* lens, void* base,
                        const g4_tile_ref* tiles, int32_t* status) {
  g4_band_desc band;
  int rc = tile_list_band(elem_type, tile_rows, tile_cols, n_tiles, tiles, &band);
  if (rc != G4_OK) return rc;
  if (!ctx) return G4_ERR_ARG;
  ctx->arenaLimit = arena_len;
  rc = decode_tiles_impl(ctx, codecs, &band, mem_space, arena, offsets, lens, base, tiles, status);
  ctx->arenaLimit = ~0ull;
  return rc;
}

int g4_decode_tiles_bounded(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space, const uint8_t* arena,
                            uint64_t arena_len, const uint64_t* offsets, const uint32_t* lens, void* grid, int32_t* status) {
  if (!ctx) return G4_ERR_ARG;
  ctx->arenaLimit = arena_len;
  const int rc = g4_decode_tiles(ctx, codecs, band, mem_space, arena, offsets, lens, grid, status);
  ctx->arenaLimit = ~0ull;
  return rc;
}

// ---- integer-coded float elements ------------------------------------------------------------------------------------
static bool icf_valid(const g4_icf_desc* icf) { return icf && icf->scale != 0.0f && std::isfinite(icf->scale); }
static g4::IcfMap icf_of(const g4_icf_desc* icf) { return g4::IcfMap{icf->scale, icf->offset, icf->fill_int, icf->fill_value}; }
struct IcfScope {  // the descriptor is valid for one call only
  g4_context* c;
  IcfScope(g4_context* ctx, const g4_icf_desc* icf) : c(ctx) { c->icfOn = true; c->icf = icf_of(icf); }
  ~IcfScope() { c->icfOn = false; c->icf = g4::IcfMap{}; }
};

int g4_icf_map(g4_context* ctx, int to_float, const g4_icf_desc* icf, int mem_space, int64_t n_rows, int64_t n_cols, const void* src,
               int64_t src_pitch, void* dst, int64_t dst_pitch) {
  if (!ctx || !icf_valid(icf) || !src || !dst || n_rows < 1 || n_cols < 1 || src_pitch < n_cols || dst_pitch < n_cols) return G4_ERR_ARG;
  ENTER(ctx);
  const g4::IcfMap m = icf_of(icf);
  if (mem_space == G4_MEM_DEVICE) {
    CK(launch_icf_map(to_float, src, src_pitch, dst, dst_pitch, n_rows, n_cols, m, ctx->stream));
    ctx->launches++;
    return G4_OK;
  }
  if (mem_space != G4_MEM_HOST) return G4_ERR_ARG;
  const size_t rowBytes = size_t(n_cols) * 4;
  CK(ctx->sGrid.ensure(rowBytes * size_t(n_rows)));
  CK(cudaMemcpy2DAsync(ctx->sGrid.p, rowBytes, src, size_t(src_pitch) * 4, rowBytes, size_t(n_rows), cudaMemcpyHostToDevice, ctx->stream));
  CK(launch_icf_map(to_float, ctx->sGrid.p, n_cols, ctx->sGrid.p, n_cols, n_rows, n_cols, m, ctx->stream));
  ctx->launches++;
  CK(cudaMemcpy2DAsync(dst, size_t(dst_pitch) * 4, ctx->sGrid.p, rowBytes, rowBytes, size_t(n_rows), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return G4_OK;
}

int g4_encode_tiles_icf(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, const g4_icf_desc* icf, int mem_space,
                        const float* grid, uint8_t* arena, uint64_t arena_cap, uint64_t* offsets, uint32_t* lens, uint8_t* codec_out,
                        uint8_t* predictor_out, int32_t* status, uint64_t* total_bytes) {
  if (!ctx || !band || band->elem_type != G4_ELEM_ICF || !icf_valid(icf)) return G4_ERR_ARG;
  IcfScope scope(ctx, icf);
  return encode_tiles_impl(ctx, codecs, band, mem_space, grid, nullptr, arena, arena_cap, offsets, lens, codec_out, predictor_out, status,
                           total_bytes);
}

int g4_decode_tiles_icf(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, const g4_icf_desc* icf, int mem_space,
                        const uint8_t* arena, uint64_t arena_len, const uint64_t* offsets, const uint32_t* lens, float* grid,
                        int32_t* status) {
  if (!ctx || !band || band->elem_type != G4_ELEM_ICF || !icf_valid(icf)) return G4_ERR_ARG;
  IcfScope scope(ctx, icf);
  return g4_decode_tiles_bounded(ctx, codecs, band, mem_space, arena, arena_len, offsets, lens, grid, status);
}

// ---- window reads: GvrsElement.readBlock (gvrs/GvrsElement.java:298-404) on the device ----------------------------------
// gather (window tiles' payload locations) -> classify + decoders -> store.  A tile-aligned window is decoded straight into
// `out` and the store launch only fills absent tiles; any other window is decoded into an int32 staging band of its covering
// tiles (4 bytes per sample) and the store launch crops, converts and fills in one pass.  Launches beyond those of
// g4_decode_tiles_bounded on the same tiles: exactly two (gather, store).
int g4_decode_window(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* raster, const g4_icf_desc* icf, const uint8_t* image,
                     uint64_t image_len, const uint64_t* payload_offsets, const uint32_t* lens, const int32_t* tile_status, uint32_t fill_bits,
                     int64_t row0, int64_t col0, int64_t n_rows, int64_t n_cols, void* out, int64_t out_pitch, int32_t* status) {
  if (!ctx || !codecs || !image || !payload_offsets || !lens || !tile_status || !out || !status) return G4_ERR_ARG;
  int rc = check_band(raster, icf != nullptr);
  if (rc != G4_OK) return rc;
  if (icf && !icf_valid(icf)) return G4_ERR_ARG;
  const int R = raster->tile_rows, Cc = raster->tile_cols;
  const int64_t gridRows = int64_t(raster->tiles_down) * R, gridCols = int64_t(raster->tiles_across) * Cc;
  if (n_rows < 1 || n_cols < 1 || row0 < 0 || col0 < 0 || row0 > gridRows - n_rows || col0 > gridCols - n_cols) return G4_ERR_ARG;
  if (out_pitch < n_cols) return G4_ERR_ARG;
  g4_codec_list ids;
  int opts[G4_MAX_CODECS];
  if (split_codec_list(codecs, &ids, opts) != G4_OK) return G4_ERR_ARG;
  codecs = &ids;
  ENTER(ctx);
  const int tr0 = int(row0 / R), tc0 = int(col0 / Cc);
  const int nTd = int((row0 + n_rows - 1) / R) - tr0 + 1, nTa = int((col0 + n_cols - 1) / Cc) - tc0 + 1;
  const int nW = nTd * nTa;
  CK(ctx->winOff.ensure(size_t(nW) * 8));
  CK(ctx->winLen.ensure(size_t(nW) * 4));
  CK(ctx->winAbsent.ensure(size_t(nW)));
  CK(launch_window_gather(payload_offsets, lens, tile_status, raster->tiles_across, tr0, tc0, nTd, nTa, ctx->winOff.as<uint64_t>(),
                          ctx->winLen.as<uint32_t>(), ctx->winAbsent.as<uint8_t>(), ctx->stream));
  ctx->launches++;
  struct ArenaScope {  // payloads that leave the image are G4_ERR_FORMAT, as in g4_decode_tiles_bounded
    g4_context* c;
    ~ArenaScope() { c->arenaLimit = ~0ull; }
  } arenaScope{ctx};
  ctx->arenaLimit = image_len;
  WindowStore ws{};
  ws.rows = n_rows;
  ws.cols = n_cols;
  ws.out = out;
  ws.outPitch = out_pitch;
  ws.R = R;
  ws.C = Cc;
  ws.nTa = nTa;
  ws.nW = nW;
  ws.absent = ctx->winAbsent.as<uint8_t>();
  ws.status = status;
  ws.fillBits = fill_bits;
  ws.mode = raster->elem_type == G4_ELEM_I16 ? kWindowNarrow16 : icf ? kWindowIcfFloat : kWindowCopy32;
  if (icf) ws.icf = icf_of(icf);
  g4_band_desc b = *raster;
  b.tiles_down = nTd;
  b.tiles_across = nTa;
  if (row0 % R == 0 && col0 % Cc == 0 && n_rows == int64_t(nTd) * R && n_cols == int64_t(nTa) * Cc) {
    b.grid_pitch = out_pitch;
    if (icf) {
      IcfScope scope(ctx, icf);
      rc = decode_device(ctx, codecs, &b, image, ctx->winOff.as<uint64_t>(), ctx->winLen.as<uint32_t>(), out, status);
    } else {
      rc = decode_device(ctx, codecs, &b, image, ctx->winOff.as<uint64_t>(), ctx->winLen.as<uint32_t>(), out, status);
    }
  } else {
    b = widened(b);  // int32 samples, pitch = the covering tiles' width
    if (raster->elem_type == G4_ELEM_F32) b.elem_type = G4_ELEM_F32;
    CK(ctx->winStage.ensure(band_samples(b) * 4));
    rc = decode_device_i32(ctx, codecs, &b, image, ctx->winOff.as<uint64_t>(), ctx->winLen.as<uint32_t>(), ctx->winStage.p, status,
                           raster->elem_type == G4_ELEM_I16);
    ws.stage = ctx->winStage.as<int32_t>();
    ws.stagePitch = b.grid_pitch;
    ws.sr0 = row0 - int64_t(tr0) * R;
    ws.sc0 = col0 - int64_t(tc0) * Cc;
  }
  if (rc != G4_OK) return rc;
  CK(launch_window_store(ws, ctx->smCount, ctx->stream));
  ctx->launches++;
  if (ctx->asyncDevice) return G4_OK;  // enqueued; status[] is read by the caller after g4_context_synchronize
  std::vector<int32_t> st(nW);
  CK(cudaMemcpyAsync(st.data(), status, size_t(nW) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int32_t& s : st)
    if (s == G4_DECLINED) s = G4_OK;  // absent tiles read as fill values; they are neither errors nor notes
  return first_bad_status(st);
}

// ---- per-tile entry points: one-tile bands through the same kernels --------------------------------

static int encode_one(g4_context* ctx, int codec_id, int codec_index, int elem, int n_rows, int n_cols, const void* values,
                      uint8_t* out, size_t out_cap, size_t* out_len, int* predictor) {
  if (!ctx || !values || !out || !out_len) return G4_ERR_ARG;
  int opts = 0;
  if (split_codec_id(codec_id, &codec_id, &opts) != G4_OK) return G4_ERR_ARG;
  if (codec_id < 0 || codec_id >= G4_CODEC_COUNT || codec_index < 0 || codec_index > 255) return G4_ERR_ARG;
  if (codec_is_float(codec_id) != (elem == G4_ELEM_F32)) return G4_DECLINED;  // e.g. CodecHuffman.encodeFloats -> null
  if (codec_id == G4_CODEC_LSOP08) return G4_DECLINED;  // decode-only legacy codec (include/g4codec.h)
  g4_band_desc band{elem, n_rows, n_cols, 1, 1, n_cols};
  int rc = check_band(&band);
  // a shape the kernels do not take (a one-row / one-column tile, more than 2^20 samples): the codec declines like a
  // reference codec that returns null, and CodecMaster / TileElement store the tile raw (ICompressionEncoder.java:61)
  if (rc == G4_ERR_UNSUPPORTED) return G4_DECLINED;
  if (rc != G4_OK) return rc;
  ENTER(ctx);
  const size_t n = size_t(n_rows) * n_cols;
  const size_t slotBytes = round_up(n * 6 + 1024, 16);  // worst case of any codec stream for this tile
  CK(ctx->sGrid.ensure(n * 4));
  CK(ctx->slots[0].ensure(slotBytes));
  CK(ctx->candLens.ensure(4));
  CK(ctx->candPreds.ensure(1));
  CK(ctx->candStatus.ensure(4));
  CK(ctx->counters.ensure(64 * sizeof(int)));
  CK(cudaMemsetAsync(ctx->counters.p, 0, 64 * sizeof(int), ctx->stream));
  CK(cudaMemcpyAsync(ctx->sGrid.p, values, n * 4, cudaMemcpyHostToDevice, ctx->stream));
  EncodeArgs a{};
  a.band = band;
  a.grid = ctx->sGrid.p;
  a.slots = ctx->slots[0].as<uint8_t>();
  a.slotBytes = slotBytes;
  a.lens = ctx->candLens.as<uint32_t>();
  a.preds = ctx->candPreds.as<uint8_t>();
  a.status = ctx->candStatus.as<int32_t>();
  a.counter = ctx->counters.as<int>();
  a.codecIndex = codec_index;
  rc = launch_encoder(ctx, codec_id, opts, a, 1);
  if (rc != G4_OK) return rc;
  uint32_t len = 0;
  int32_t st = 0;
  uint8_t pred = 0;
  CK(cudaMemcpyAsync(&len, a.lens, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(&st, a.status, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(&pred, a.preds, 1, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (st == G4_ERR_CAPACITY) return G4_DECLINED;  // a packing that outgrows its slot is longer than the raw tile anyway
  if (st != G4_OK) return st;
  *out_len = len;
  if (predictor) *predictor = pred;
  if (len > out_cap) return G4_ERR_CAPACITY;
  CK(cudaMemcpyAsync(out, a.slots, len, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return G4_OK;
}

static int decode_one(g4_context* ctx, int codec_id, int elem, int n_rows, int n_cols, const uint8_t* packing, size_t len, void* out) {
  if (!ctx || !packing || !out || len == 0 || len > 0xffffffffull) return G4_ERR_ARG;
  int opts = 0;  // ignored, as in g4_decode_tiles
  if (split_codec_id(codec_id, &codec_id, &opts) != G4_OK) return G4_ERR_ARG;
  if (codec_id < 0 || codec_id >= G4_CODEC_COUNT) return G4_ERR_ARG;
  if (codec_is_float(codec_id) != (elem == G4_ELEM_F32)) return G4_DECLINED;  // decodeFloats on an int codec -> null
  g4_band_desc band{elem, n_rows, n_cols, 1, 1, n_cols};
  int rc = check_band(&band);
  if (rc != G4_OK) return rc;
  ENTER(ctx);
  const size_t n = size_t(n_rows) * n_cols;
  CK(ctx->sGrid.ensure(n * 4));
  CK(ctx->sArena.ensure(len + 16));
  CK(ctx->sOffsets.ensure(8));
  CK(ctx->sLens.ensure(4));
  CK(ctx->sStatus.ensure(4));
  CK(ctx->lists.ensure(4));
  CK(ctx->counters.ensure(64 * sizeof(int)));
  const size_t stride = round_up(n * 6 + 64, 16);
  CK(ctx->scratch.ensure(stride));
  CK(cudaMemsetAsync(ctx->counters.p, 0, 64 * sizeof(int), ctx->stream));
  CK(cudaMemsetAsync(ctx->sOffsets.p, 0, 8, ctx->stream));
  CK(cudaMemsetAsync(ctx->lists.p, 0, 4, ctx->stream));
  const uint32_t len32 = uint32_t(len);
  const int one = 1;
  const int32_t pending = 99;  // positive sentinel: a kernel that never reports leaves an unknown status
  CK(cudaMemcpyAsync(ctx->sArena.p, packing, len, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->sLens.p, &len32, 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->counters.as<int>() + 32, &one, 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->sStatus.p, &pending, 4, cudaMemcpyHostToDevice, ctx->stream));
  DecodeArgs a{};
  a.band = band;
  a.grid = ctx->sGrid.p;
  a.arena = ctx->sArena.as<uint8_t>();
  a.offsets = ctx->sOffsets.as<uint64_t>();
  a.lens = ctx->sLens.as<uint32_t>();
  a.list = ctx->lists.as<int>();
  a.listCount = ctx->counters.as<int>() + 32;
  a.status = ctx->sStatus.as<int32_t>();
  a.counter = ctx->counters.as<int>() + 16;
  a.scratch = ctx->scratch.as<uint8_t>();
  a.scratchStride = stride;
  rc = launch_decoder(ctx, codec_id, a, 1);
  if (rc != G4_OK) return rc;
  int32_t st = 0;
  CK(cudaMemcpyAsync(&st, ctx->sStatus.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (st != G4_OK && st != G4_CHECKSUM_MISMATCH) return st;
  CK(cudaMemcpyAsync(out, ctx->sGrid.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return st;  // G4_OK, or G4_CHECKSUM_MISMATCH with the values delivered
}

// ---- ICompressionDecoder.analyze ----------------------------------------------------------------------------------------
int g4_analyze_tiles(g4_context* ctx, const g4_codec_list* codecs, const g4_band_desc* band, int mem_space, const uint8_t* arena,
                     uint64_t arena_len, const uint64_t* offsets, const uint32_t* lens, g4_tile_stats* stats, uint64_t* pair_counts) {
  if (!ctx || !codecs || !band || !arena || !offsets || !lens || !stats) return G4_ERR_ARG;
  int rc = check_band(band);
  if (rc != G4_OK) return rc;
  g4_codec_list ids;  // the option bits are ignored, as in decode
  int opts[G4_MAX_CODECS];
  if (split_codec_list(codecs, &ids, opts) != G4_OK) return G4_ERR_ARG;
  codecs = &ids;
  ENTER(ctx);
  const int nTiles = band->tiles_down * band->tiles_across;
  const size_t n = size_t(band->tile_rows) * band->tile_cols;
  const int nCtas = persistent_ctas(ctx, nTiles, 4);
  const size_t stride = round_up(n * 6 + 64, 16);
  CK(ctx->scratch.ensure(stride * nCtas));
  AnalyzeArgs a{};
  a.nTiles = nTiles;
  a.nCells = uint32_t(n);
  a.rawLen = standard_size(*band);
  a.codecs = *codecs;
  a.scratch = ctx->scratch.as<uint8_t>();
  a.scratchStride = stride;
  constexpr size_t kPairBytes = size_t(2) * 5 * 65536 * 8;
  if (mem_space == G4_MEM_DEVICE) {
    a.arena = arena;
    a.arenaLen = arena_len;
    a.offsets = offsets;
    a.lens = lens;
    a.stats = stats;
    a.pairs = reinterpret_cast<unsigned long long*>(pair_counts);
    CK(launch_analyze(a, nCtas, ctx->stream));
    ctx->launches++;
    CK(cudaStreamSynchronize(ctx->stream));
    return G4_OK;
  }
  if (mem_space != G4_MEM_HOST) return G4_ERR_ARG;
  uint64_t arenaBytes = 0;
  std::vector<uint64_t> off(offsets, offsets + nTiles);
  std::vector<uint32_t> ln(lens, lens + nTiles);
  for (int t = 0; t < nTiles; t++) {
    if (off[size_t(t)] > arena_len || ln[size_t(t)] > arena_len - off[size_t(t)]) { off[size_t(t)] = 0; ln[size_t(t)] = 0; }  // -> G4_ERR_FORMAT for the tile
    arenaBytes = std::max<uint64_t>(arenaBytes, off[size_t(t)] + ln[size_t(t)]);
  }
  CK(ctx->sArena.ensure(arenaBytes + 16));
  CK(ctx->sOffsets.ensure(size_t(nTiles) * 8));
  CK(ctx->sLens.ensure(size_t(nTiles) * 4));
  CK(ctx->sGrid.ensure(round_up(size_t(nTiles) * sizeof(g4_tile_stats), 16) + (pair_counts ? kPairBytes : 0)));
  CK(cudaMemcpyAsync(ctx->sArena.p, arena, arenaBytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->sOffsets.p, off.data(), size_t(nTiles) * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->sLens.p, ln.data(), size_t(nTiles) * 4, cudaMemcpyHostToDevice, ctx->stream));
  uint8_t* dPairs = ctx->sGrid.as<uint8_t>() + round_up(size_t(nTiles) * sizeof(g4_tile_stats), 16);
  if (pair_counts) CK(cudaMemcpyAsync(dPairs, pair_counts, kPairBytes, cudaMemcpyHostToDevice, ctx->stream));
  a.arena = ctx->sArena.as<uint8_t>();
  a.arenaLen = arenaBytes;
  a.offsets = ctx->sOffsets.as<uint64_t>();
  a.lens = ctx->sLens.as<uint32_t>();
  a.stats = ctx->sGrid.as<g4_tile_stats>();
  a.pairs = pair_counts ? reinterpret_cast<unsigned long long*>(dPairs) : nullptr;
  CK(launch_analyze(a, nCtas, ctx->stream));
  ctx->launches++;
  CK(cudaMemcpyAsync(stats, a.stats, size_t(nTiles) * sizeof(g4_tile_stats), cudaMemcpyDeviceToHost, ctx->stream));
  if (pair_counts) CK(cudaMemcpyAsync(pair_counts, dPairs, kPairBytes, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return G4_OK;
}

// ---- predictor models on their own (IPredictorModel.java:42-173) ---------------------------------------------------
int g4_predictor_tiles(g4_context* ctx, int model, int int_flavour, int decode, const g4_band_desc* band, void* grid, uint8_t* slots,
                       uint64_t slot_bytes, uint32_t* lens, int32_t* seeds, int32_t* status) {
  if (!ctx || !band || !grid || !slots || !lens || !seeds || !status) return G4_ERR_ARG;
  if (model < G4_PRED_DIFFERENCING || model > G4_PRED_DIFF_NULLS || band->elem_type != G4_ELEM_I32) return G4_ERR_ARG;
  int rc = check_band(band);
  if (rc != G4_OK) return rc;
  const uint64_t n = uint64_t(band->tile_rows) * uint64_t(band->tile_cols);
  if ((slot_bytes & 15) != 0 || slot_bytes < (int_flavour ? 4 * n : 6 * n + 16) || (reinterpret_cast<uintptr_t>(slots) & 15) != 0) return G4_ERR_ARG;
  ENTER(ctx);
  PredictorArgs a{};
  a.band = *band;
  a.grid = grid;
  a.model = model;
  a.intFlavour = int_flavour ? 1 : 0;
  a.slots = slots;
  a.slotBytes = size_t(slot_bytes);
  a.lens = lens;
  a.seeds = seeds;
  a.status = status;
  const int nTiles = band->tiles_down * band->tiles_across;
  CK(launch_predictor(a, decode, persistent_ctas(ctx, nTiles, 8), ctx->stream));
  ctx->launches++;
  return G4_OK;
}

static int predictor_one(g4_context* ctx, int model, int int_flavour, int decode, int32_t* seed, int n_rows, int n_cols, int32_t* values,
                         void* stream, size_t stream_cap, size_t* n_stream) {
  if (!ctx || !values || !stream || !seed || !n_stream) return G4_ERR_ARG;
  g4_band_desc band{G4_ELEM_I32, n_rows, n_cols, 1, 1, n_cols};
  int rc = check_band(&band);
  if (rc == G4_ERR_UNSUPPORTED && !decode) return G4_DECLINED;
  if (rc != G4_OK) return rc;
  ENTER(ctx);
  const size_t n = size_t(n_rows) * n_cols;
  const size_t slotBytes = round_up(n * 6 + 64, 16);
  CK(ctx->sGrid.ensure(n * 4));
  CK(ctx->scratch.ensure(slotBytes));
  CK(ctx->sLens.ensure(4));
  CK(ctx->sStatus.ensure(4));
  CK(ctx->sOffsets.ensure(8));
  uint32_t len32 = 0;
  if (decode) {
    const size_t bytes = int_flavour ? *n_stream * 4 : *n_stream;
    if (bytes + 16 > slotBytes || *n_stream > 0xffffffffull) return G4_ERR_FORMAT;
    len32 = uint32_t(*n_stream);
    CK(cudaMemsetAsync(ctx->scratch.p, 0, slotBytes, ctx->stream));
    CK(cudaMemcpyAsync(ctx->scratch.p, stream, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->sLens.p, &len32, 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->sOffsets.p, seed, 4, cudaMemcpyHostToDevice, ctx->stream));
  } else CK(cudaMemcpyAsync(ctx->sGrid.p, values, n * 4, cudaMemcpyHostToDevice, ctx->stream));
  rc = g4_predictor_tiles(ctx, model, int_flavour, decode, &band, ctx->sGrid.p, ctx->scratch.as<uint8_t>(), slotBytes, ctx->sLens.as<uint32_t>(),
                          ctx->sOffsets.as<int32_t>(), ctx->sStatus.as<int32_t>());
  if (rc != G4_OK) return rc;
  int32_t st = 0;
  CK(cudaMemcpyAsync(&st, ctx->sStatus.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(&len32, ctx->sLens.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (!decode) CK(cudaMemcpyAsync(seed, ctx->sOffsets.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (st != G4_OK) return st;
  if (decode) CK(cudaMemcpyAsync(values, ctx->sGrid.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  else {
    const size_t bytes = int_flavour ? size_t(len32) * 4 : size_t(len32);
    *n_stream = len32;
    if (bytes > stream_cap) return G4_ERR_CAPACITY;
    CK(cudaMemcpyAsync(stream, ctx->scratch.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return G4_OK;
}

int g4_predictor_encode(g4_context* ctx, int model, int n_rows, int n_cols, const int32_t* values, int32_t* seed, uint8_t* m32_out,
                        size_t out_cap, size_t* n_bytes) {
  return predictor_one(ctx, model, 0, 0, seed, n_rows, n_cols, const_cast<int32_t*>(values), m32_out, out_cap, n_bytes);
}
int g4_predictor_encode_int(g4_context* ctx, int model, int n_rows, int n_cols, const int32_t* values, int32_t* seed, int32_t* residuals_out,
                            size_t out_cap, size_t* n_residuals) {
  return predictor_one(ctx, model, 1, 0, seed, n_rows, n_cols, const_cast<int32_t*>(values), residuals_out, out_cap * 4, n_residuals);
}
int g4_predictor_decode(g4_context* ctx, int model, int32_t seed, int n_rows, int n_cols, const uint8_t* m32, size_t n_bytes, int32_t* values_out) {
  return predictor_one(ctx, model, 0, 1, &seed, n_rows, n_cols, values_out, const_cast<uint8_t*>(m32), 0, &n_bytes);
}
int g4_predictor_decode_int(g4_context* ctx, int model, int32_t seed, int n_rows, int n_cols, const int32_t* residuals, size_t n_residuals,
                            int32_t* values_out) {
  return predictor_one(ctx, model, 1, 1, &seed, n_rows, n_cols, values_out, const_cast<int32_t*>(residuals), 0, &n_residuals);
}

int g4_encode_i32(g4_context* ctx, int codec_id, int codec_index, int n_rows, int n_cols, const int32_t* values, uint8_t* out,
                  size_t out_cap, size_t* out_len, int* predictor) {
  return encode_one(ctx, codec_id, codec_index, G4_ELEM_I32, n_rows, n_cols, values, out, out_cap, out_len, predictor);
}
int g4_decode_i32(g4_context* ctx, int codec_id, int n_rows, int n_cols, const uint8_t* packing, size_t len, int32_t* out) {
  return decode_one(ctx, codec_id, G4_ELEM_I32, n_rows, n_cols, packing, len, out);
}
int g4_encode_f32(g4_context* ctx, int codec_id, int codec_index, int n_rows, int n_cols, const float* values, uint8_t* out,
                  size_t out_cap, size_t* out_len) {
  return encode_one(ctx, codec_id, codec_index, G4_ELEM_F32, n_rows, n_cols, values, out, out_cap, out_len, nullptr);
}
int g4_decode_f32(g4_context* ctx, int codec_id, int n_rows, int n_cols, const uint8_t* packing, size_t len, float* out) {
  return decode_one(ctx, codec_id, G4_ELEM_F32, n_rows, n_cols, packing, len, out);
}

}  // extern "C"
