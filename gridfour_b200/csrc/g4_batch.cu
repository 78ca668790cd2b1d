// g4_batch.cu -- the selection layer and data-movement kernels around the codec kernels.
//
// Reference semantics reproduced here (paths under /root/reference/core/src/main/java/org/gridfour/):
//   CodecMaster.encodeSingleThread  gvrs/CodecMaster.java:150-169   strictly smallest, ties -> lowest index
//   TileElementInt.encode/decode    gvrs/TileElementInt.java:196-219  raw little-endian when len >= 4n
//   CodecMaster.decode              gvrs/CodecMaster.java:195-203   dispatch on packing[0]
#include "g4_kernels.h"
#include "g4_device.cuh"
#include "../../include/g4terrain.h"

namespace g4 {

__global__ void fill_terrain_kernel(int elemType, uint64_t seed, int64_t row0, int64_t col0, int64_t nRows, int64_t nCols,
                                    void* out) {
  const int64_t total = nRows * nCols;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    int64_t r = i / nCols, c = i - r * nCols;
    if (elemType == G4_ELEM_I32) static_cast<int32_t*>(out)[i] = g4_terrain_m(seed, row0 + r, col0 + c);
    else static_cast<float*>(out)[i] = float(g4_terrain_dm(seed, row0 + r, col0 + c)) * 0.1f;
  }
}

// Best-of selection.  cand arrays are [nCand][nTiles]; candIndex[c] = codec list position of candidate c
// (ascending, so the first strictly-smallest candidate is the lowest index).
__global__ void select_kernel(SelectArgs a) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.nTiles) return;
  uint32_t best = 0xffffffffu;
  int bc = -1;
  int st = G4_OK;
  for (int c = 0; c < a.nCand; c++) {
    int s = a.candStatus[size_t(c) * a.nTiles + t];
    uint32_t l = a.candLens[size_t(c) * a.nTiles + t];
    if (s == G4_OK && l > 0 && l < best) { best = l; bc = c; }
    else if (s < 0 && s != G4_ERR_CAPACITY && st == G4_OK) st = s;  // a candidate failed (not "declined")
  }
  const uint32_t rawLen = a.rawLen;
  if (bc < 0 || best >= rawLen) {  // TileElementInt.java:198-204
    a.lens[t] = rawLen;
    a.codecOut[t] = G4_CODEC_RAW;
    a.predOut[t] = 0;
    a.src[t] = -1;
  } else {
    a.lens[t] = best;
    a.codecOut[t] = uint8_t(a.candIndex[bc]);
    a.predOut[t] = a.candPreds[size_t(bc) * a.nTiles + t];
    a.src[t] = bc;
  }
  a.status[t] = st;
}

// Exclusive scan of the 8-byte-aligned payload lengths -> offsets; one CTA.
__global__ void __launch_bounds__(kThreads) offsets_kernel(const uint32_t* lens, uint64_t* offsets, int nTiles, uint64_t* total) {
  __shared__ unsigned long long sm[kWarps];
  __shared__ unsigned long long carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int t0 = 0; t0 < nTiles; t0 += kThreads) {
    int t = t0 + threadIdx.x;
    unsigned long long x = t < nTiles ? ((unsigned long long)(lens[t]) + 7ull) & ~7ull : 0ull;
    unsigned long long inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      unsigned long long y = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += y;
    }
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    unsigned long long base = carry;
    for (int w = 0; w < warp; w++) base += sm[w];
    if (t < nTiles) offsets[t] = base + inc - x;
    __syncthreads();
    if (threadIdx.x == kThreads - 1) carry = base + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

// One CTA per tile: copy the winner's packing (or the raw samples) to arena + offsets[t].
// Destination offsets are multiples of 8; the tail of the last 8-byte word is zero filled.
__global__ void __launch_bounds__(kThreads) compact_kernel(CompactArgs a) {
  const int t = blockIdx.x;
  const uint32_t len = a.lens[t];
  const uint64_t off = a.offsets[t];
  if (off + ((uint64_t(len) + 7) & ~7ull) > a.arenaCap) {
    if (threadIdx.x == 0) a.status[t] = G4_ERR_CAPACITY;
    return;
  }
  uint8_t* dst = a.arena + off;
  const int src = a.src[t];
  if (src < 0 && a.raw16) {  // TileElementShort raw form: little-endian shorts, zero padded to a multiple of 4 bytes
    const int R = a.band.tile_rows, C = a.band.tile_cols, n = R * C;
    const int tr = t / a.band.tiles_across, tc = t - tr * a.band.tiles_across;
    const int16_t* base = a.raw16 + int64_t(tr) * R * a.raw16Pitch + int64_t(tc) * C;
    uint32_t* d32 = reinterpret_cast<uint32_t*>(dst);
    const int nWords = int((len + 3u) >> 2);
    for (int i = threadIdx.x; i < ((nWords + 1) & ~1); i += kThreads) {
      uint32_t w = 0;
      for (int h = 0; h < 2; h++) {
        int k = 2 * i + h;
        if (k < n) { int r = k / C, c = k - r * C; w |= uint32_t(uint16_t(base[int64_t(r) * a.raw16Pitch + c])) << (16 * h); }
      }
      d32[i] = w;
    }
  } else if (src < 0) {
    const TileView tv = tile_view(a.band, a.grid, t);
    uint32_t* d32 = reinterpret_cast<uint32_t*>(dst);
    const int n = tv.R * tv.C;
    for (int i = threadIdx.x; i < n; i += kThreads) {
      int r = i / tv.C, c = i - r * tv.C;
      d32[i] = uint32_t(tv.at(r, c));
    }
    if ((n & 1) && threadIdx.x == 0) d32[n] = 0;
  } else {
    const uint32_t* s32 = reinterpret_cast<const uint32_t*>(a.slots[src] + size_t(t) * a.slotBytes);
    uint32_t* d32 = reinterpret_cast<uint32_t*>(dst);
    const uint32_t nWords = ((len + 7u) & ~7u) >> 2;
    for (uint32_t i = threadIdx.x; i < nWords; i += kThreads) {
      uint32_t w = 0;
      if (i * 4u < len) {
        w = s32[i];
        uint32_t valid = len - i * 4u;
        if (valid < 4u) w &= (1u << (8u * valid)) - 1u;
      }
      d32[i] = w;
    }
  }
}

// Decode-side classification: one thread per tile appends the tile to the list of its codec kind.
// lists layout: [G4_CODEC_COUNT + 1][nTiles]; kind G4_CODEC_COUNT == raw.
__global__ void classify_kernel(ClassifyArgs a) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.nTiles) return;
  const uint32_t len = a.lens[t];
  int kind;
  int st = G4_OK;
  // a payload must lie inside the arena; one longer than the raw tile is never written (TileElementInt.encode :196-205
  // stores the raw samples instead) and would overflow the decoders' per-tile bounds
  if (len > a.rawLen || a.offsets[t] > a.arenaLen || uint64_t(len) > a.arenaLen - a.offsets[t]) { kind = -1; st = G4_ERR_FORMAT; }
  else if (len == a.rawLen) kind = G4_CODEC_COUNT;
  else if (len == 0) { kind = -1; st = G4_ERR_FORMAT; }
  else {
    int index = a.arena[a.offsets[t]];
    if (index >= a.codecs.n_codecs) { kind = -1; st = G4_ERR_FORMAT; }  // CodecMaster.java:197-199
    else {
      kind = a.codecs.codec_ids[index];
      bool isFloatCodec = kind == G4_CODEC_FLOAT;
      if (kind < 0 || kind >= G4_CODEC_COUNT || isFloatCodec != (a.elemType == G4_ELEM_F32)) { kind = -1; st = G4_ERR_FORMAT; }
    }
  }
  a.status[t] = st;
  if (kind >= 0) {
    int pos = atomicAdd(&a.counts[kind], 1);
    a.lists[size_t(kind) * a.nTiles + pos] = t;
  }
}

__global__ void __launch_bounds__(kThreads) raw_decode_kernel(DecodeArgs a) {
  const int li = blockIdx.x;
  if (li >= *a.listCount) return;
  const int t = a.list[li];
  const TileView tv = tile_view(a.band, a.grid, t);
  const uint8_t* src = a.arena + a.offsets[t];
  const int n = tv.R * tv.C;
  if (a.rawShorts) {
    for (int i = threadIdx.x; i < n; i += kThreads) {
      int r = i / tv.C, c = i - r * tv.C;
      tv.at(r, c) = int32_t(int16_t(uint16_t(src[2 * size_t(i)]) | (uint16_t(src[2 * size_t(i) + 1]) << 8)));
    }
    return;
  }
  const bool aligned = (reinterpret_cast<uintptr_t>(src) & 3) == 0;
  for (int i = threadIdx.x; i < n; i += kThreads) {
    int r = i / tv.C, c = i - r * tv.C;
    uint32_t v = aligned ? reinterpret_cast<const uint32_t*>(src)[i] : load_le32(src + 4 * size_t(i));
    tv.at(r, c) = int32_t(v);
  }
}

// TileElementShort.encode (:213-220): widen, fill value -> INT4_NULL_CODE
__global__ void widen_i16_kernel(const int16_t* src, int64_t srcPitch, int32_t* dst, int64_t rows, int64_t cols, int32_t fill) {
  const int64_t total = rows * cols;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    int64_t r = i / cols, c = i - r * cols;
    int32_t v = src[r * srcPitch + c];
    dst[i] = v == fill ? kNull : v;
  }
}
// TileElementShort.decode (:236-245): INT4_NULL_CODE -> SHORT_NULL_CODE, everything else narrowed with a (short) cast
__global__ void narrow_i16_kernel(const int32_t* src, int16_t* dst, int64_t dstPitch, int64_t rows, int64_t cols) {
  const int64_t total = rows * cols;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    int64_t r = i / cols, c = i - r * cols;
    int32_t v = src[i];
    dst[r * dstPitch + c] = v == kNull ? int16_t(-32768) : int16_t(v);
  }
}

// Integer-coded float elements (GvrsElementSpecificationIntCodedFloat / GvrsElementIntCodedFloat).  The reference source
// is not in this tree; these are the formulas as the ICF feature request restates them (the oracle's g4o_icf.cpp states
// them once more).  No reference fixture pins them beyond exactly representable values.
//   float -> code: NaN -> fillInt; else (int) Math.floor((double)((v - offset) * scale) + 0.5): float32 subtract and multiply,
//                  correctly rounded and not fused, + 0.5 and floor in double, Java's saturating (int) cast (NaN -> 0),
//                  which is what PTX cvt.rzi.s32.f64 does.
//   code -> float: fillInt -> fillValue; else (float) code / scale + offset in float32, with a true IEEE division.
__device__ __forceinline__ int32_t icf_code(float v, const IcfMap& m) {
  if (v != v) return m.fillInt;
  return __double2int_rz(floor(__dadd_rn(double(__fmul_rn(__fsub_rn(v, m.offset), m.scale)), 0.5)));
}
__device__ __forceinline__ float icf_value(int32_t k, const IcfMap& m) {
  return k == m.fillInt ? m.fillValue : __fadd_rn(__fdiv_rn(__int2float_rn(k), m.scale), m.offset);
}
__device__ __forceinline__ int32_t icf_apply(float v, const IcfMap& m) { return icf_code(v, m); }
__device__ __forceinline__ float icf_apply(int32_t k, const IcfMap& m) { return icf_value(k, m); }

// One pass over a pitched rows x cols rectangle (pitches in samples); src and dst may be the same buffer.  Each thread maps
// four consecutive cells of a row: with one 16-byte load and store where both row starts are 16-byte aligned, cell by cell
// otherwise (pitches or offsets that are not multiples of 4, and the last partial quad of a row).  blockDim = (bx, 256 / bx)
// with bx sized to the row, so that narrow rectangles keep the threads busy; no division per cell.
template <class S, class D, class S4, class D4>
__device__ __forceinline__ void icf_map_rect(const S* src, int64_t srcPitch, D* dst, int64_t dstPitch, int64_t rows, int64_t cols,
                                             const IcfMap& m) {
  const int64_t c = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (c >= cols) return;
  for (int64_t r = int64_t(blockIdx.y) * blockDim.y + threadIdx.y; r < rows; r += int64_t(gridDim.y) * blockDim.y) {
    const S* s = src + r * srcPitch + c;
    D* d = dst + r * dstPitch + c;
    if (c + 4 <= cols && ((reinterpret_cast<uintptr_t>(s) | reinterpret_cast<uintptr_t>(d)) & 15) == 0) {
      const S4 x = *reinterpret_cast<const S4*>(s);
      D4 y;
      y.x = icf_apply(x.x, m);
      y.y = icf_apply(x.y, m);
      y.z = icf_apply(x.z, m);
      y.w = icf_apply(x.w, m);
      *reinterpret_cast<D4*>(d) = y;
    } else {
      const int k = cols - c < 4 ? int(cols - c) : 4;
      for (int i = 0; i < k; i++) d[i] = icf_apply(s[i], m);
    }
  }
}
__global__ void __launch_bounds__(256) icf_to_int_kernel(const float* src, int64_t srcPitch, int32_t* dst, int64_t dstPitch, int64_t rows,
                                                         int64_t cols, IcfMap m) {
  icf_map_rect<float, int32_t, float4, int4>(src, srcPitch, dst, dstPitch, rows, cols, m);
}
__global__ void __launch_bounds__(256) icf_to_float_kernel(const int32_t* src, int64_t srcPitch, float* dst, int64_t dstPitch,
                                                           int64_t rows, int64_t cols, IcfMap m) {
  icf_map_rect<int32_t, float, int4, float4>(src, srcPitch, dst, dstPitch, rows, cols, m);
}

// ---- window reads (g4_decode_window, GvrsElement.readBlock :298-404) ------------------------------------------------------
// One thread per window tile: the tile's payload location in window order.  Tiles the file does not hold (G4_DECLINED) and
// damaged records (< 0) get a zero-length payload, which classify_kernel puts in no decoder list.
__global__ void window_gather_kernel(const uint64_t* offsets, const uint32_t* lens, const int32_t* tileStatus, int tilesAcross, int tr0,
                                     int tc0, int nTd, int nTa, uint64_t* offW, uint32_t* lenW, uint8_t* absentW) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nTd * nTa) return;
  const int wr = w / nTa, wc = w - wr * nTa;
  const int64_t t = int64_t(tr0 + wr) * tilesAcross + (tc0 + wc);
  const int32_t st = tileStatus[t];
  offW[w] = st == G4_OK ? offsets[t] : 0;
  lenW[w] = st == G4_OK ? lens[t] : 0u;
  absentW[w] = st == G4_DECLINED ? 1 : 0;
}

// classify_kernel reported the zero-length payloads of absent tiles as G4_ERR_FORMAT; they are G4_DECLINED, not errors.
__device__ __forceinline__ void window_mark_absent(const WindowStore& a) {
  const int64_t nThreads = int64_t(gridDim.x) * gridDim.y * blockDim.x * blockDim.y;
  const int64_t id = (int64_t(blockIdx.y) * gridDim.x + blockIdx.x) * (blockDim.x * blockDim.y) + threadIdx.y * blockDim.x + threadIdx.x;
  for (int64_t w = id; w < a.nW; w += nThreads)
    if (a.absent[w]) a.status[w] = G4_DECLINED;
}

template <int Mode> struct WindowOut { using T = int32_t; using V = int4; };
template <> struct WindowOut<kWindowNarrow16> { using T = int16_t; using V = short4; };
template <> struct WindowOut<kWindowIcfFloat> { using T = float; using V = float4; };

template <int Mode>
__device__ __forceinline__ typename WindowOut<Mode>::T window_sample(int32_t v, const WindowStore& a) {
  if constexpr (Mode == kWindowNarrow16) return v == kNull ? int16_t(-32768) : int16_t(v);  // as narrow_i16_kernel
  else if constexpr (Mode == kWindowIcfFloat) return icf_value(v, a.icf);
  else return v;
}
template <int Mode>
__device__ __forceinline__ typename WindowOut<Mode>::T window_fill(const WindowStore& a) {
  if constexpr (Mode == kWindowNarrow16) return int16_t(uint16_t(a.fillBits));
  else if constexpr (Mode == kWindowIcfFloat) return __uint_as_float(a.fillBits);
  else return int32_t(a.fillBits);
}

// The store pass of an unaligned window: staging band -> the caller's rectangle, cropped, converted, absent tiles filled.
// Threads take four consecutive cells of a row as icf_map_rect does: one 16-byte load where the staging address is 16-byte
// aligned, one 16-byte (8-byte for shorts) store where the output address is, cell by cell otherwise.
template <int Mode>
__global__ void __launch_bounds__(256) window_store_kernel(WindowStore a) {
  using T = typename WindowOut<Mode>::T;
  using V = typename WindowOut<Mode>::V;
  window_mark_absent(a);
  const int64_t c = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (c >= a.cols) return;
  const int k = a.cols - c < 4 ? int(a.cols - c) : 4;
  const int64_t sc = a.sc0 + c;
  const int tcA = int(sc / a.C), tcB = int((sc + k - 1) / a.C);  // window tile columns of the first and last cell
  const T fill = window_fill<Mode>(a);
  for (int64_t r = int64_t(blockIdx.y) * blockDim.y + threadIdx.y; r < a.rows; r += int64_t(gridDim.y) * blockDim.y) {
    const int64_t sr = a.sr0 + r;
    const uint8_t* absentRow = a.absent + (sr / a.R) * a.nTa;
    const int32_t* s = a.stage + sr * a.stagePitch + sc;
    T* d = static_cast<T*>(a.out) + r * a.outPitch + c;
    int32_t v[4] = {0, 0, 0, 0};
    if (k == 4 && (reinterpret_cast<uintptr_t>(s) & 15) == 0) {
      const int4 x = *reinterpret_cast<const int4*>(s);
      v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; i++)
        if (i < k) v[i] = s[i];
    }
    T y[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const bool gone = i < k && absentRow[tcA == tcB ? tcA : int((sc + i) / a.C)];
      y[i] = gone ? fill : window_sample<Mode>(v[i], a);
    }
    if (k == 4 && (reinterpret_cast<uintptr_t>(d) & (sizeof(V) - 1)) == 0) {
      V z;
      z.x = y[0]; z.y = y[1]; z.z = y[2]; z.w = y[3];
      *reinterpret_cast<V*>(d) = z;
    } else {
#pragma unroll
      for (int i = 0; i < 4; i++)
        if (i < k) d[i] = y[i];
    }
  }
}

// A tile-aligned window decoded straight into the caller's rectangle: only absent tiles are written, with the fill sample.
template <class T>
__global__ void __launch_bounds__(256) window_fill_kernel(WindowStore a) {
  const T fill = T(a.fillBits);
  for (int w = blockIdx.x; w < a.nW; w += gridDim.x) {
    if (!a.absent[w]) continue;
    if (threadIdx.x == 0 && threadIdx.y == 0) a.status[w] = G4_DECLINED;
    const int wr = w / a.nTa, wc = w - wr * a.nTa;
    T* base = static_cast<T*>(a.out) + int64_t(wr) * a.R * a.outPitch + int64_t(wc) * a.C;
    for (int r = threadIdx.y; r < a.R; r += blockDim.y)
      for (int c = threadIdx.x; c < a.C; c += blockDim.x) base[int64_t(r) * a.outPitch + c] = fill;
  }
}

cudaError_t launch_window_gather(const uint64_t* offsets, const uint32_t* lens, const int32_t* tileStatus, int tilesAcross, int tr0,
                                 int tc0, int nTd, int nTa, uint64_t* offW, uint32_t* lenW, uint8_t* absentW, cudaStream_t s) {
  const int n = nTd * nTa;
  window_gather_kernel<<<(n + 255) / 256, 256, 0, s>>>(offsets, lens, tileStatus, tilesAcross, tr0, tc0, nTd, nTa, offW, lenW, absentW);
  return cudaGetLastError();
}
cudaError_t launch_window_store(const WindowStore& a, int smCount, cudaStream_t s) {
  if (!a.stage) {
    const int n = a.nW < smCount * 8 ? a.nW : smCount * 8;
    int bx = 32;
    while (bx < 256 && bx < a.C) bx <<= 1;
    const dim3 block(bx, 256 / bx);
    if (a.mode == kWindowNarrow16) window_fill_kernel<uint16_t><<<n, block, 0, s>>>(a);
    else window_fill_kernel<uint32_t><<<n, block, 0, s>>>(a);
    return cudaGetLastError();
  }
  const int64_t quads = (a.cols + 3) / 4;
  int bx = 1;
  while (bx < 256 && bx < quads) bx <<= 1;
  const dim3 block(bx, 256 / bx);
  const int64_t gx = (quads + bx - 1) / bx, gy = (a.rows + block.y - 1) / block.y;
  if (gx > 0x7fffffff) return cudaErrorInvalidValue;
  const dim3 grid(unsigned(gx), unsigned(gy < 65535 ? gy : 65535));
  switch (a.mode) {
    case kWindowNarrow16: window_store_kernel<kWindowNarrow16><<<grid, block, 0, s>>>(a); break;
    case kWindowIcfFloat: window_store_kernel<kWindowIcfFloat><<<grid, block, 0, s>>>(a); break;
    default: window_store_kernel<kWindowCopy32><<<grid, block, 0, s>>>(a); break;
  }
  return cudaGetLastError();
}

cudaError_t launch_fill_terrain(int elemType, uint64_t seed, int64_t row0, int64_t col0, int64_t nRows, int64_t nCols, void* out,
                                cudaStream_t s) {
  fill_terrain_kernel<<<148 * 8, 256, 0, s>>>(elemType, seed, row0, col0, nRows, nCols, out);
  return cudaGetLastError();
}
cudaError_t launch_widen_i16(const int16_t* src, int64_t srcPitch, int32_t* dst, int64_t rows, int64_t cols, int32_t fill, cudaStream_t s) {
  widen_i16_kernel<<<148 * 8, 256, 0, s>>>(src, srcPitch, dst, rows, cols, fill);
  return cudaGetLastError();
}
cudaError_t launch_narrow_i16(const int32_t* src, int16_t* dst, int64_t dstPitch, int64_t rows, int64_t cols, cudaStream_t s) {
  narrow_i16_kernel<<<148 * 8, 256, 0, s>>>(src, dst, dstPitch, rows, cols);
  return cudaGetLastError();
}
cudaError_t launch_icf_map(int toFloat, const void* src, int64_t srcPitch, void* dst, int64_t dstPitch, int64_t rows, int64_t cols,
                           const IcfMap& m, cudaStream_t s) {
  const int64_t quads = (cols + 3) / 4;
  int bx = 1;
  while (bx < 256 && bx < quads) bx <<= 1;
  const dim3 block(bx, 256 / bx);
  const int64_t gx = (quads + bx - 1) / bx, gy = (rows + block.y - 1) / block.y;
  if (gx > 0x7fffffff) return cudaErrorInvalidValue;
  const dim3 grid(unsigned(gx), unsigned(gy < 65535 ? gy : 65535));
  if (toFloat)
    icf_to_float_kernel<<<grid, block, 0, s>>>(static_cast<const int32_t*>(src), srcPitch, static_cast<float*>(dst), dstPitch, rows, cols, m);
  else
    icf_to_int_kernel<<<grid, block, 0, s>>>(static_cast<const float*>(src), srcPitch, static_cast<int32_t*>(dst), dstPitch, rows, cols, m);
  return cudaGetLastError();
}
cudaError_t launch_select(const SelectArgs& a, cudaStream_t s) {
  select_kernel<<<(a.nTiles + 255) / 256, 256, 0, s>>>(a);
  return cudaGetLastError();
}
cudaError_t launch_offsets(const uint32_t* lens, uint64_t* offsets, int nTiles, uint64_t* total, cudaStream_t s) {
  offsets_kernel<<<1, kThreads, 0, s>>>(lens, offsets, nTiles, total);
  return cudaGetLastError();
}
cudaError_t launch_compact(const CompactArgs& a, int nTiles, cudaStream_t s) {
  compact_kernel<<<nTiles, kThreads, 0, s>>>(a);
  return cudaGetLastError();
}
cudaError_t launch_classify(const ClassifyArgs& a, cudaStream_t s) {
  classify_kernel<<<(a.nTiles + 255) / 256, 256, 0, s>>>(a);
  return cudaGetLastError();
}
cudaError_t launch_raw_decode(const DecodeArgs& a, int nTiles, cudaStream_t s) {
  raw_decode_kernel<<<nTiles, kThreads, 0, s>>>(a);
  return cudaGetLastError();
}

}  // namespace g4
