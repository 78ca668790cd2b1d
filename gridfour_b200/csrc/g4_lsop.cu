// g4_lsop.cu -- LSOP12 (Lewis-Smith optimal predictor, 12 coefficients) on sm_100a.
//
// Reference (under /root/reference/core/src/main/java/org/gridfour/lsop/):
//   LsDecoder12.java:94-470 (decode, unpackInitializers, unpackInterior), LsHeader.java:104-265,
//   LsOptimalPredictor12.java:109-383, LsEncoder12.java:122-219
//
// Decode is two kernels over the LSOP tiles of a band:
//   A  one CTA per tile: header parse, entropy stage (canonical Huffman type 2, legacy Huffman + M32 type 0)
//      with residuals scattered to their raster cells, then rows 0/1 and columns 0/1 by prefix scans;
//   B  one WARP per tile: the causal 12-tap float32 stencil is nonlinear (rounding), so it cannot be a scan.
//      Cells with equal c+3r are independent: lane l owns row r0+l and runs three columns behind lane l-1.
//      Row r-1/r-2 operands travel between lanes by warp shuffles; the two last columns of every row
//      (Triangle predictor) ride the same schedule.  Float arithmetic is strictly left to right, no FMA.
#include <utility>
#include "g4_kernels.h"
#include "g4_predict.cuh"
#include "g4_huffdec.cuh"
#include "g4_canon.cuh"
#include "g4_canon_fast.cuh"
#include "g4_canon_enc.cuh"
#include "g4_inflate.cuh"
#include "g4_m32stream.cuh"
#include "g4_lsop_common.cuh"

namespace g4 {

namespace {

union LsopDecShared {
  HuffDecShared h;
  CanonDecShared c;
  InflateWarpShared inf;
};


struct CellSink {
  TileView t;
  int order;
  __device__ __forceinline__ void operator()(uint32_t k, int32_t v) const {
    int r, c;
    stream_to_cell(order, int(k), t.R, t.C, &r, &c);
    t.at(r, c) = v;
  }
};

struct InteriorRunSink {  // LSOP12 interior order: rows 2.., columns 2..C-3 row-major; running cell address, no division per value
  static constexpr bool kPacked = false;
  TileView t;
  int32_t* p;  // column 2 of the current row
  int c, w;
  __device__ __forceinline__ void begin(uint32_t k0) {
    w = t.C - 4;
    int rr = int(k0) / w;
    c = int(k0) - rr * w;
    p = t.row(2 + rr) + 2;
  }
  __device__ __forceinline__ void put(int32_t v) {
    p[c] = v;
    if (++c == w) { c = 0; p += t.pitch; }
  }
  __device__ __forceinline__ void end() {}
};
// Packed form for 16-byte aligned tile rows (canon_fast_decode_text, Sink::kPacked): the symbol bytes (value + 128) of
// every lookup are appended to a register byte queue; whenever the queue covers the rest of the current 8-column group
// (32-byte sector) the group leaves as two int4 stores -- bytes to ints by one XOR per four bytes and one sign-extending
// PRMT per value.  Only the 6-column groups at both ends of a row's interior (columns 2..7 and C-8..C-3), the unaligned
// head and the tail of a run, and the rare values (escapes, nulls) take the scalar path.
// prmt with the sign-replicating selector nibbles (8 | byte index); __byte_perm masks that bit away
__device__ __forceinline__ int32_t sx_byte(uint32_t x, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(x), "r"(0u), "r"(sel));
  return int32_t(d);
}
struct InteriorPackedSink {
  static constexpr bool kPacked = true;
  TileView t;
  int32_t* rowp;  // column 0 of the current row
  int col;        // next column to be written (2 .. C-3)
  int cnt, need;  // queued bytes; bytes that complete the current group (cnt < need between calls)
  uint64_t lo;    // queue bytes 0..7, oldest in the low byte
  uint32_t hi;    // queue bytes 8..9
  __device__ __forceinline__ int group_need() const {
    const int a = 8 - (col & 7), b = t.C - 2 - col;
    return a < b ? a : b;
  }
  __device__ __forceinline__ void begin(uint32_t k0) {
    const int w = t.C - 4;
    const int rr = int(k0) / w;
    col = 2 + int(k0) - rr * w;
    rowp = t.row(2 + rr);
    cnt = 0;
    lo = 0;
    hi = 0;
    need = group_need();
  }
  __device__ __forceinline__ void advance_group() {
    if (col == t.C - 2) { col = 2; rowp += t.pitch; }
    need = group_need();
  }
  __device__ __forceinline__ void write_scalars(int k) {  // the k oldest queue bytes, k <= cnt <= 9, inside the current group
    const uint32_t x0 = uint32_t(lo) ^ 0x80808080u, x1 = uint32_t(lo >> 32) ^ 0x80808080u;
    int32_t* const q = rowp + col;
    if (k > 0) q[0] = sx_byte(x0, 0x8880);
    if (k > 1) q[1] = sx_byte(x0, 0x9991);
    if (k > 2) q[2] = sx_byte(x0, 0xaaa2);
    if (k > 3) q[3] = sx_byte(x0, 0xbbb3);
    if (k > 4) q[4] = sx_byte(x1, 0x8880);
    if (k > 5) q[5] = sx_byte(x1, 0x9991);
    if (k > 6) q[6] = sx_byte(x1, 0xaaa2);
    if (k > 7) q[7] = sx_byte(x1, 0xbbb3);
    if (k > 8) q[8] = int32_t(hi & 0xffu) - 128;
    drop(k);
    col += k;
  }
  __device__ __forceinline__ void drop(int k) {  // removes the k oldest queue bytes (k <= 9)
    const int sh = 8 * k;
    if (k >= 8) { lo = uint64_t(hi) >> (sh - 64); hi = 0; }
    else if (k > 0) { lo = (lo >> sh) | (uint64_t(hi) << (64 - sh)); hi = 0; }  // hi holds at most 2 bytes: they all move into lo
    cnt -= k;
  }
  __device__ __forceinline__ void flush() {
    do {
      const int ph = col & 7;
      if (need == 8) {
        // the common case, an aligned group of eight: no variable shifts, the two leftover bytes move down
        const uint32_t x0 = uint32_t(lo) ^ 0x80808080u, x1 = uint32_t(lo >> 32) ^ 0x80808080u;
        int32_t* const g = rowp + col;
        *reinterpret_cast<int4*>(g) = make_int4(sx_byte(x0, 0x8880), sx_byte(x0, 0x9991), sx_byte(x0, 0xaaa2), sx_byte(x0, 0xbbb3));
        *reinterpret_cast<int4*>(g + 4) = make_int4(sx_byte(x1, 0x8880), sx_byte(x1, 0x9991), sx_byte(x1, 0xaaa2), sx_byte(x1, 0xbbb3));
        lo = hi;
        hi = 0;
        cnt -= 8;
        col += 8;
      } else if (need == 6 && (ph == 0 || ph == 2)) {
        // an aligned group of eight, or the six-column group at either end of a row's interior (columns 2..7 as
        // int2 + int4, columns C-8..C-3 as int4 + int2): queue byte j goes to column col + j
        const uint64_t al = lo << (8 * ph);
        const uint32_t x0 = uint32_t(al) ^ 0x80808080u, x1 = uint32_t(al >> 32) ^ 0x80808080u;
        int32_t* const g = rowp + (col - ph);
        if (ph == 0) *reinterpret_cast<int4*>(g) = make_int4(sx_byte(x0, 0x8880), sx_byte(x0, 0x9991), sx_byte(x0, 0xaaa2), sx_byte(x0, 0xbbb3));
        else *reinterpret_cast<int2*>(g + 2) = make_int2(sx_byte(x0, 0xaaa2), sx_byte(x0, 0xbbb3));
        if (ph + need == 8) *reinterpret_cast<int4*>(g + 4) = make_int4(sx_byte(x1, 0x8880), sx_byte(x1, 0x9991), sx_byte(x1, 0xaaa2), sx_byte(x1, 0xbbb3));
        else *reinterpret_cast<int2*>(g + 4) = make_int2(sx_byte(x1, 0x8880), sx_byte(x1, 0x9991));
        const int k = need;
        drop(k);
        col += k;
      } else write_scalars(need);
      advance_group();
    } while (cnt >= need);
  }
  __device__ __forceinline__ void push(uint32_t bytes, int n) {  // n = 1..3 symbol bytes, first value in the low byte
    const int sh = cnt * 8;  // cnt <= 7
    lo |= uint64_t(bytes) << sh;
    if (sh > 40) hi |= bytes >> (64 - sh);
    cnt += n;
    if (cnt >= need) flush();
  }
  __device__ __forceinline__ void put_rare(int32_t v) {
    write_scalars(cnt);
    rowp[col] = v;
    col++;
    advance_group();
  }
  // an escape extends the value before it (CanonicalHuffman.java:495-504): v = (v << nb) | bits, in place
  __device__ __forceinline__ void amend(int nb, uint32_t bits) {
    write_scalars(cnt);
    need = group_need();
    int32_t* cell = col > 2 ? rowp + col - 1 : rowp - t.pitch + (t.C - 3);
    *cell = int32_t((uint32_t(*cell) << nb) | bits);
  }
  __device__ __forceinline__ void end() { write_scalars(cnt); }
};

}  // namespace

// LsDecoder12.unpackInitializers (:204-241): row 0 and column 0 by differencing, row 1 and column 1 by Triangle.
// Precondition: every initializer cell holds its residual.  All threads call.
__device__ inline void lsop_init_scans(const TileView& t, int32_t seed) {
  __shared__ uint32_t scan[kWarps + 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int R = t.R, C = t.C;
  __syncthreads();
  if (tid == 0) t.at(0, 0) = seed;
  __syncthreads();
  if (warp == 0) row_scan_warp(t.row(0), C, 0);
  column0_scan(t, scan);  // ends with __syncthreads
  if (warp == 0) {
    // row 1: T[c] = v[1][c] - v[0][c];  T[c] = T[c-1] + residual(1,c)
    uint32_t carry = uint32_t(t.at(1, 0)) - uint32_t(t.at(0, 0));
    for (int c0 = 1; c0 < C; c0 += 32) {
      int c = c0 + lane;
      uint32_t x = c < C ? uint32_t(t.at(1, c)) : 0u;
      uint32_t inc = warp_inclusive_scan(x);
      if (c < C) t.at(1, c) = int32_t(carry + inc + uint32_t(t.at(0, c)));
      carry += __shfl_sync(0xffffffffu, inc, 31);
    }
  }
  __syncthreads();
  {
    // column 1, rows 2..: U[r] = v[r][1] - v[r][0];  U[r] = U[r-1] + residual(r,1)
    uint32_t carry = uint32_t(t.at(1, 1)) - uint32_t(t.at(1, 0));
    for (int r0 = 2; r0 < R; r0 += kThreads) {
      int r = r0 + tid;
      uint32_t x = r < R ? uint32_t(t.at(r, 1)) : 0u;
      uint32_t tot;
      uint32_t ex = block_exclusive_scan(x, scan, &tot);
      if (r < R) t.at(r, 1) = int32_t(carry + ex + x + uint32_t(t.at(r, 0)));
      carry += tot;
    }
  }
}

// ---- kernel A, fast path: canonical-Huffman packings (type 2) ------------------------------------------------------
// Two kernels, so that no CTA ever waits on a serial table parse:
//   H  one WARP per tile: LSOP header, both canonical code tables, the short initializer stream (decoded serially
//      by lane 0 -- ~1200 values -- while the other warps of the SM work on their own tiles), rows 0,1 / columns 0,1 by
//      warp scans.  Exports the interior stream's 260 code lengths and text position to `meta`.
//   T  one CTA per tile: the interior text (the bulk of the bits) with the staged sub-sequence decoder of
//      g4_canon_fast.cuh; no serial section.
// Legacy-Huffman, Deflate, oversized or unaligned packings are appended to `defer` for the general kernel below.

// Column scan by one warp: cell (r0-1, c) holds a final value, cells (r, c) r >= r0 hold d[r]; after the call
// v[r][c] = base[r] + (carry0 + d[r0] + ... + d[r]) with base[r] = v[r][c-1] when addLeft, else 0.
__device__ inline void lsop_warp_column_scan(const TileView& t, int col, int r0, uint32_t carry, bool addLeft) {
  const int lane = threadIdx.x & 31;
  for (int rb = r0; rb < t.R; rb += 32) {
    const int r = rb + lane;
    uint32_t x = r < t.R ? uint32_t(t.at(r, col)) : 0u;
    uint32_t inc = warp_inclusive_scan(x);
    if (r < t.R) t.at(r, col) = int32_t(carry + inc + (addLeft ? uint32_t(t.at(r, col - 1)) : 0u));
    carry += __shfl_sync(0xffffffffu, inc, 31);
  }
  __syncwarp();
}

__global__ void __launch_bounds__(kThreads, 5) lsop_decode_head_kernel(DecodeArgs a, float* coefOut, uint8_t* meta, int* defer,
                                                                    int* deferCount, uint32_t stageWords) {
  __shared__ CanonWarpShared WS[kWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  CanonWarpShared& W = WS[warp];
  const int li = blockIdx.x * kWarps + warp;
  if (li >= *a.listCount) return;
  const int tIdx = a.list[li];
  uint8_t* m = meta + size_t(tIdx) * kLsopMetaBytes;
  if (lane == 0) *reinterpret_cast<uint32_t*>(m) = 0;
  const TileView t = tile_view(a.band, a.grid, tIdx);
  const int R = t.R, C = t.C;
  const uint8_t* packing = a.arena + a.offsets[tIdx];
  const uint32_t len = a.lens[tIdx];
  LsHeaderInfo h = parse_ls_header(packing, len, coefOut + size_t(tIdx) * 12, lane == 0);
  if (lane == 0 && a.lsopCks && h.ok && h.hasChecksum) { a.lsopCks[2 * tIdx] = 1u; a.lsopCks[2 * tIdx + 1] = h.valueChecksum; }
  if (!h.ok || R < 6 || C < 6) {
    if (lane == 0) a.status[tIdx] = G4_ERR_FORMAT;
    return;
  }
  if (h.type != 2 || len > stageWords * 4u || (reinterpret_cast<uintptr_t>(packing) & 3) != 0) {
    if (lane == 0) defer[atomicAdd(deferCount, 1)] = tIdx;
    return;
  }
  const uint32_t nInit = uint32_t(4 * R + 2 * C - 9);
  BitSrc src;
  src.init(packing, len);  // absolute bit positions inside the packing
  canon_warp_parse_header(W, src, h.headerSize * 8u);
  int status = W.error ? G4_ERR_FORMAT : G4_OK;
  uint32_t endBit = 0;
  if (status == G4_OK) {
    // initializer text (CanonicalHuffman.decodeText :469-519), ~1200 values: warp-level sub-sequence decode, every
    // lane scatters the values it decoded to the cells of the initializer stream order
    uint32_t eb = 0, nv = 0;
    auto emit = [&](uint32_t k, int32_t v) {
      int r, c;
      stream_to_cell(kStreamLsopInit, int(k), R, C, &r, &c);
      t.at(r, c) = v;
    };
    const bool ok = canon_warp_decode_text(W, src, W.textStart, nInit, emit, &eb, &nv) && nv == nInit;
    __syncwarp();
    if (lane == 0) {
      if (!ok) W.error = 1;
      W.textStart = eb;
    }
    __syncwarp();
    if (W.error) status = G4_ERR_FORMAT;
    endBit = W.textStart;
  }
  if (status == G4_OK) {
    canon_warp_parse_header(W, src, endBit);  // interior stream: tables only, exported for kernel T
    if (W.error) status = G4_ERR_FORMAT;
    else {
      for (int i = lane; i < kCanonSymbols; i += 32) m[8 + i] = W.lens[i];
      if (lane == 0) *reinterpret_cast<uint32_t*>(m) = W.textStart;
    }
  }
  if (status == G4_OK) {
    // LsDecoder12.unpackInitializers (:204-241): row 0 and column 0 by differencing, row 1 and column 1 by Triangle
    if (lane == 0) t.at(0, 0) = h.seed;
    __syncwarp();
    row_scan_warp(t.row(0), C, 0);
    __syncwarp();
    lsop_warp_column_scan(t, 0, 1, uint32_t(h.seed), false);
    {
      // row 1: T[c] = v[1][c] - v[0][c];  T[c] = T[c-1] + residual(1,c)
      uint32_t carry = uint32_t(t.at(1, 0)) - uint32_t(t.at(0, 0));
      for (int c0 = 1; c0 < C; c0 += 32) {
        int c = c0 + lane;
        uint32_t x = c < C ? uint32_t(t.at(1, c)) : 0u;
        uint32_t inc = warp_inclusive_scan(x);
        if (c < C) t.at(1, c) = int32_t(carry + inc + uint32_t(t.at(0, c)));
        carry += __shfl_sync(0xffffffffu, inc, 31);
      }
    }
    __syncwarp();
    // column 1, rows 2..: U[r] = v[r][1] - v[r][0];  U[r] = U[r-1] + residual(r,1)
    lsop_warp_column_scan(t, 1, 2, uint32_t(t.at(1, 1)) - uint32_t(t.at(1, 0)), true);
  }
  if (lane == 0) a.status[tIdx] = status;
}

template <class InteriorSink>
__global__ void __launch_bounds__(kThreads, 4) lsop_decode_text_kernel(DecodeArgs a, const uint8_t* meta) {
  extern __shared__ __align__(16) unsigned char lsopFastSmem[];
  CanonFastShared& F = *reinterpret_cast<CanonFastShared*>(lsopFastSmem);
  __shared__ int sTile;
  const int tid = threadIdx.x;
  for (;;) {
    __syncthreads();
    if (tid == 0) sTile = atomicAdd(a.counter, 1);
    __syncthreads();
    const int li = sTile;
    if (li >= *a.listCount) break;
    const int tIdx = a.list[li];
    const uint8_t* m = meta + size_t(tIdx) * kLsopMetaBytes;
    const uint32_t T0 = *reinterpret_cast<const uint32_t*>(m);
    if (T0 == 0) continue;  // deferred or rejected by kernel H
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const uint8_t* packing = a.arena + a.offsets[tIdx];
    const uint32_t len = a.lens[tIdx];
    const uint32_t nInterior = uint32_t(t.R - 2) * uint32_t(t.C - 4);
    canon_fast_stage(F, packing, len);
    for (int i = tid; i < kCanonSymbols; i += kThreads) F.lens[i] = m[8 + i];
    if (tid == 0) F.error = 0;
    __syncthreads();
    canon_fast_tables_cta(F);
    bool ok = F.error == 0;
    if (ok) {
      canon_fast_build_lut(F);
      uint32_t endBit = 0, nv = 0;
      InteriorSink s2{};
      s2.t = t;
      ok = canon_fast_decode_text(F, len * 8u, T0, nInterior, 0u, s2, &endBit, &nv) && nv == nInterior;
    }
    if (!ok && tid == 0) a.status[tIdx] = G4_ERR_FORMAT;
  }
}

// ---- kernel A ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) lsop_decode_entropy_kernel(DecodeArgs a, float* coefOut) {
  __shared__ LsopDecShared S;
  __shared__ int sTile;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (;;) {
    __syncthreads();
    if (tid == 0) sTile = atomicAdd(a.counter, 1);
    __syncthreads();
    const int li = sTile;
    if (li >= *a.listCount) break;
    const int tIdx = a.list[li];
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int R = t.R, C = t.C;
    const uint8_t* packing = a.arena + a.offsets[tIdx];
    const uint32_t len = a.lens[tIdx];
    int status = G4_OK;
    LsHeaderInfo h = parse_ls_header(packing, len, coefOut + size_t(tIdx) * 12, tid == 0);
    if (tid == 0 && a.lsopCks && h.ok && h.hasChecksum) { a.lsopCks[2 * tIdx] = 1u; a.lsopCks[2 * tIdx + 1] = h.valueChecksum; }
    const uint32_t nInit = uint32_t(4 * R + 2 * C - 9);
    const uint32_t nInterior = uint32_t(R - 2) * uint32_t(C - 4);
    if (!h.ok || R < 6 || C < 6) status = G4_ERR_FORMAT;
    if (status == G4_OK) {
      BitSrc src;
      src.init(packing + h.headerSize, len - h.headerSize);
      if (h.type == 2) {
        uint32_t endBit = 0, nv = 0;
        CellSink s1{t, kStreamLsopInit};
        CellSink s2{t, kStreamLsopInterior};
        if (!canon_decode_stream(S.c, src, 0, nInit, 32768u, s1, &endBit, &nv) || nv != nInit) status = G4_ERR_FORMAT;
        else if (!canon_decode_stream(S.c, src, endBit, nInterior, 0u, s2, &endBit, &nv) || nv != nInterior) status = G4_ERR_FORMAT;
      } else {
        // type 0: two legacy Huffman streams back to back, each M32 coded (LsDecoder12.java:119-124)
        // type 1: two zlib streams; the second starts where the first one's input ended (:126-145)
        if (h.nInitCodes < nInit || h.nInitCodes > 6 * nInit || h.nInteriorCodes < nInterior || h.nInteriorCodes > 6 * nInterior)
          status = G4_ERR_FORMAT;
        else {
          uint8_t* m32a = a.scratch + size_t(blockIdx.x) * a.scratchStride;
          uint8_t* m32b = m32a + ((size_t(h.nInitCodes) + 31) & ~size_t(15));
          uint32_t endBit = 0;
          bool entropyOk;
          if (h.type == 1) {
            __shared__ int sInfOk;
            if (warp == 0) {
              const uint8_t* z = packing + h.headerSize;
              const uint32_t zLen = len - h.headerSize;
              uint32_t produced = 0, consumed = 0;
              int rc = inflate_warp(S.inf, z, zLen, m32a, h.nInitCodes, &produced, &consumed);
              bool ok = rc == kInfOk && produced == h.nInitCodes && consumed <= zLen;
              if (ok) {
                uint32_t c1 = consumed;
                rc = inflate_warp(S.inf, z + c1, zLen - c1, m32b, h.nInteriorCodes, &produced, &consumed);
                ok = rc == kInfOk && produced == h.nInteriorCodes;
              }
              if (lane == 0) sInfOk = ok ? 1 : 0;
            }
            __syncthreads();
            entropyOk = sInfOk != 0;
          } else {
            entropyOk = huffman_decode_stream(S.h, src, 0, h.nInitCodes, m32a, &endBit) &&
                        huffman_decode_stream(S.h, src, endBit, h.nInteriorCodes, m32b, &endBit);
          }
          if (!entropyOk) status = G4_ERR_FORMAT;
          else {
            __syncthreads();
            __shared__ uint32_t scanM[kWarps + 1];
            if (!m32_parse_to_cells(m32a, h.nInitCodes, kStreamLsopInit, t, nInit, scanM)) status = G4_ERR_FORMAT;
            else if (!m32_parse_to_cells(m32b, h.nInteriorCodes, kStreamLsopInterior, t, nInterior, scanM)) status = G4_ERR_FORMAT;
          }
        }
      }
    }
    if (status == G4_OK) lsop_init_scans(t, h.seed);
    __syncthreads();
    if (tid == 0) a.status[tIdx] = status;
  }
}

// ---- LSOP08: the legacy 8-coefficient codec (decode only) ------------------------------------------------------------
// lsop/LsDecoder08.java:65-163.  Same header class as LSOP12 (eight coefficients), legacy Huffman or two zlib streams over
// M32 bytes, other initializers (rows 0 and 1 whole, columns 0 and 1 of the rest), an 8-tap stencil that only looks up and
// left, and the estimate is (int)(p + 0.5f) -- float addition, then truncation -- instead of StrictMath.round.
// The reference no longer registers this codec (lsop/LsCodecUtility.java:73), so it gets the plain general form.
__global__ void __launch_bounds__(kThreads) lsop08_decode_entropy_kernel(DecodeArgs a, float* coefOut) {
  __shared__ LsopDecShared S;
  __shared__ int sTile;
  __shared__ uint32_t scanM[kWarps + 1];
  __shared__ int sInfOk;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (;;) {
    __syncthreads();
    if (tid == 0) sTile = atomicAdd(a.counter, 1);
    __syncthreads();
    const int li = sTile;
    if (li >= *a.listCount) break;
    const int tIdx = a.list[li];
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int R = t.R, C = t.C;
    const uint8_t* packing = a.arena + a.offsets[tIdx];
    const uint32_t len = a.lens[tIdx];
    int status = G4_OK;
    LsHeaderInfo h = parse_ls_header(packing, len, coefOut + size_t(tIdx) * 12, tid == 0, 8);
    const uint32_t nInit = uint32_t((C - 1) + C + 2 * (R - 2));
    const uint32_t nInterior = uint32_t(R - 2) * uint32_t(C - 2);
    if (!h.ok || R < 3 || C < 3) status = G4_ERR_FORMAT;
    else if (h.nInitCodes < nInit || h.nInitCodes > 6 * nInit || h.nInteriorCodes < nInterior || h.nInteriorCodes > 6 * nInterior)
      status = G4_ERR_FORMAT;
    if (status == G4_OK) {
      uint8_t* m32a = a.scratch + size_t(blockIdx.x) * a.scratchStride;
      uint8_t* m32b = m32a + ((size_t(h.nInitCodes) + 31) & ~size_t(15));
      bool entropyOk;
      if (h.type != 0) {  // LsDecoder08.java:83-105: everything but type 0 is two zlib streams
        if (warp == 0) {
          const uint8_t* z = packing + h.headerSize;
          const uint32_t zLen = len - h.headerSize;
          uint32_t produced = 0, consumed = 0;
          int rc = inflate_warp(S.inf, z, zLen, m32a, h.nInitCodes, &produced, &consumed);
          bool ok = rc == kInfOk && produced == h.nInitCodes && consumed <= zLen;
          if (ok) {
            const uint32_t c1 = consumed;
            rc = inflate_warp(S.inf, z + c1, zLen - c1, m32b, h.nInteriorCodes, &produced, &consumed);
            ok = rc == kInfOk && produced == h.nInteriorCodes;
          }
          if (lane == 0) sInfOk = ok ? 1 : 0;
        }
        __syncthreads();
        entropyOk = sInfOk != 0;
      } else {
        BitSrc src;
        src.init(packing + h.headerSize, len - h.headerSize);
        uint32_t endBit = 0;
        entropyOk = huffman_decode_stream(S.h, src, 0, h.nInitCodes, m32a, &endBit) &&
                    huffman_decode_stream(S.h, src, endBit, h.nInteriorCodes, m32b, &endBit);
      }
      if (!entropyOk) status = G4_ERR_FORMAT;
      else {
        __syncthreads();
        if (!m32_parse_to_cells(m32a, h.nInitCodes, kStreamLsop8Init, t, nInit, scanM)) status = G4_ERR_FORMAT;
        else if (!m32_parse_to_cells(m32b, h.nInteriorCodes, kStreamLsop8Interior, t, nInterior, scanM)) status = G4_ERR_FORMAT;
      }
    }
    if (status == G4_OK) {
      // LsDecoder08.unpackInitializers (:115-135)
      __syncthreads();
      if (tid == 0) t.at(0, 0) = h.seed;
      __syncthreads();
      if (warp == 0) row_scan_warp(t.row(0), C, 0);            // v[0][c] = seed + d[1] + ... + d[c]
      if (warp == 1) row_scan_warp(t.row(1), C, 0);            // running sum of row 1's differences
      __syncthreads();
      for (int c = tid; c < C; c += kThreads) t.at(1, c) = int32_t(uint32_t(t.at(1, c)) + uint32_t(h.seed));
      __syncthreads();
      uint32_t carry = uint32_t(t.at(1, 0));                   // column 0 from row 2: v[r][0] = v[r-1][0] + d
      for (int r0 = 2; r0 < R; r0 += kThreads) {
        const int r = r0 + tid;
        const uint32_t x = r < R ? uint32_t(t.at(r, 0)) : 0u;
        uint32_t tot;
        const uint32_t ex = block_exclusive_scan(x, scanM, &tot);
        if (r < R) {
          const uint32_t v0 = carry + ex + x;
          t.at(r, 0) = int32_t(v0);
          t.at(r, 1) = int32_t(v0 + uint32_t(t.at(r, 1)));   // v[r][1] = v[r][0] + d
        }
        carry += tot;
      }
    }
    __syncthreads();
    if (tid == 0) a.status[tIdx] = status;
  }
}

// One warp per tile, lane = row, one column behind the lane above (the stencil never looks right of its own column).
__global__ void __launch_bounds__(kThreads) lsop08_wavefront_kernel(DecodeArgs a, const float* coef) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int li = blockIdx.x * kWarps + warp;
  if (li >= *a.listCount) return;
  const int tIdx = a.list[li];
  if (a.status[tIdx] != G4_OK) return;
  const TileView t = tile_view(a.band, a.grid, tIdx);
  const int R = t.R, C = t.C;
  float u[8];
#pragma unroll
  for (int i = 0; i < 8; i++) u[i] = coef[size_t(tIdx) * 12 + i];
  for (int r0 = 2; r0 < R; r0 += 32) {
    const int r = r0 + lane;
    const bool active = r < R;
    const int rr = active ? r : R - 1;
    int32_t* rowp = t.row(rr);
    const int32_t* up1 = t.row(rr - 1);
    const int32_t* up2 = t.row(rr - 2);
    float v1 = float(rowp[1]), v2 = float(rowp[0]);  // own row, columns c-1 and c-2
    const int lastLane = (R - 1 - r0) < 31 ? (R - 1 - r0) : 31;
    const int nSteps = (C - 2) + lastLane;
    __syncwarp();
    for (int s = 0; s < nSteps; s++) {
      const int c = 2 + s - lane;
      if (active && c >= 2 && c < C) {
        // rows r-1 and r-2 up to column c were finished in earlier steps (or by the previous row group)
        const float a1 = float(__ldcg(up1 + c - 1)), a0 = float(__ldcg(up1 + c)), a2 = float(__ldcg(up1 + c - 2));
        const float b2 = float(__ldcg(up2 + c - 2)), b1 = float(__ldcg(up2 + c - 1)), b0 = float(__ldcg(up2 + c));
        // LsDecoder08.java:151-159 -- evaluated left to right in float32, no fused multiply-add
        float p = u[0] * v1;
        p = p + u[1] * a1;
        p = p + u[2] * a0;
        p = p + u[3] * v2;
        p = p + u[4] * a2;
        p = p + u[5] * b2;
        p = p + u[6] * b1;
        p = p + u[7] * b0;
        const int32_t val = int32_t(uint32_t(__float2int_rz(p + 0.5f)) + uint32_t(rowp[c]));  // (int)(p + 0.5f) + residual
        rowp[c] = val;
        v2 = v1;
        v1 = float(val);
      }
      __threadfence_block();
      __syncwarp();
    }
  }
}

// ---- kernel B: wavefront ------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) lsop_wavefront_kernel(DecodeArgs a, const float* coef) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int li = blockIdx.x * kWarps + warp;
  if (li >= *a.listCount) return;
  const int tIdx = a.list[li];
  if (a.status[tIdx] != G4_OK) return;
  const TileView t = tile_view(a.band, a.grid, tIdx);
  const int R = t.R, C = t.C;
  float u[12];
#pragma unroll
  for (int i = 0; i < 12; i++) u[i] = coef[size_t(tIdx) * 12 + i];

  for (int r0 = 2; r0 < R; r0 += 32) {
    const int r = r0 + lane;
    const bool active = r < R;
    const int rr = active ? r : R - 1;  // clamp so inactive lanes read valid memory
    int32_t* rowp = t.row(rr);
    const int32_t* up1 = t.row(rr - 1);
    const int32_t* up2 = t.row(rr - 2);
    // windows positioned for column c = -1: [c-2 .. c+2] = [-3 .. 1]
    float z1 = float(rowp[1]), z6 = float(rowp[0]);
    int32_t o1 = rowp[1];
    float z7 = 0.f, z2 = 0.f, z3 = 0.f, z4 = float(up1[0]), z5 = float(up1[1]);
    int32_t i2 = 0, i3 = 0, i4 = up1[0], i5 = up1[1];
    float z8 = 0.f, z9 = 0.f, z10 = 0.f, z11 = float(up2[0]), z12 = float(up2[1]);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    int32_t lastOut = 0;
    const int lastLane = (R - 1 - r0) < 31 ? (R - 1 - r0) : 31;
    const int nSteps = C + 3 * lastLane;  // lane l works on column s - 3l at step s; the last lane ends at column C-1
    __syncwarp();
    for (int s = 0; s < nSteps; s++) {
      const int c = s - 3 * lane;
      int32_t recvA = __shfl_up_sync(0xffffffffu, lastOut, 1);
      float recvB = __shfl_up_sync(0xffffffffu, a2, 1);
      const bool shifting = c >= 0 && c < C;
      if (lane == 0 && shifting) {
        // rows r0-1 and r0-2 were finished by the previous row group (or by kernel A for rows 0,1)
        int cc = c + 2 < C ? c + 2 : C - 1;
        recvA = __ldcg(up1 + cc);
        recvB = float(__ldcg(up2 + cc));
      }
      if (shifting) {
        float fa = float(recvA);
        z7 = z2; z2 = z3; z3 = z4; z4 = z5; z5 = fa;
        i2 = i3; i3 = i4; i4 = i5; i5 = recvA;
        z8 = z9; z9 = z10; z10 = z11; z11 = z12; z12 = recvB;
        a2 = a1; a1 = a0; a0 = fa;
      }
      if (active && c >= 2 && c < C) {
        int32_t res = rowp[c];
        int32_t val;
        if (c < C - 2) {
          // LsDecoder12.java:424-438 -- evaluated left to right in float32, no fused multiply-add
          float p = u[0] * z1;
          p = p + u[1] * z2;
          p = p + u[2] * z3;
          p = p + u[3] * z4;
          p = p + u[4] * z5;
          p = p + u[5] * z6;
          p = p + u[6] * z7;
          p = p + u[7] * z8;
          p = p + u[8] * z9;
          p = p + u[9] * z10;
          p = p + u[10] * z11;
          p = p + u[11] * z12;
          val = int32_t(uint32_t(java_round(p)) + uint32_t(res));
        } else {
          // last two columns: Triangle predictor (LsDecoder12.java:459-468)
          val = int32_t(uint32_t(res) + ((uint32_t(o1) + uint32_t(i3)) - uint32_t(i2)));
        }
        rowp[c] = val;
        lastOut = val;
        z6 = z1;
        z1 = float(val);
        o1 = val;
      }
    }
    __syncwarp();
    __threadfence_block();
  }
}

// ---- kernel B, vectorised: 4-column skew, int4 traffic, row groups pipelined back to back -----------------------------
// Same recurrence and operation order as lsop_wavefront_kernel; used when every tile row is 16-byte aligned
// (tile_cols % 4 == 0, grid_pitch % 4 == 0, aligned base).  A warp walks the tile in groups of 30 rows.  Lane l runs ONE
// 4-column block behind lane l-1, so all lanes are at the same column phase: one int4 load (residuals) and one int4
// store (values) per lane and iteration, and nothing else touches memory.  Lanes 0 and 1 are FEEDERS: they own the two
// finished rows above the group (rows 0,1 from kernel H, later the rows lanes 30,31 wrote for the previous group), load
// them like any other lane and pass them through with all-zero coefficients, so every operand of a computing lane
// arrives by shuffle from the lane above it and the loop has no lane-specific loads or selects:
//   row r-1, column c+2 = lane l-1's output of two steps ago (its float history f2);
//   row r-2, column c+2 = the oldest element lane l-1 still holds of ITS row above (its av[j]);
//   columns 0,1 of both rows (needed once per row) = lane l-1's first two outputs / first two av elements of its
//   previous block, shuffled before the windows shift.
// A row takes P = max(C,136) steps so that lanes 30,31 of a group have stored a block (and passed the __syncwarp that
// ends their iteration) at least one iteration before the next group's feeders fetch it; groups need no drain.
// Three CTAs per SM on purpose.  Every lane streams its own raster row, 16 bytes per iteration, and lives off L1: the
// 128-byte line a lane touches must survive the eight iterations that consume it.  24 warps x 32 rows keep 768 lines
// live; measured on the config-3 shard: 3 CTAs/SM 1.46 ms, 4 CTAs/SM 1.49 ms, 5 CTAs/SM (1280 lines) 18 ms -- past that
// point the lines are evicted between iterations and every load becomes a scattered 32-byte DRAM access.  L1-bypassing
// loads (ld.global.cg) show the same collapse at any occupancy (16-18 ms), and so does a second load in flight per lane.
__global__ void __launch_bounds__(kThreads, 3) lsop_wavefront4_kernel(DecodeArgs a, const float* coef) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int li = blockIdx.x * kWarps + warp;
  if (li >= *a.listCount) return;
  const int tIdx = a.list[li];
  if (a.status[tIdx] != G4_OK) return;
  const TileView t = tile_view(a.band, a.grid, tIdx);
  const int R = t.R, C = t.C;
  const bool feeder = lane < 2;
  float u[12];
#pragma unroll
  for (int i = 0; i < 12; i++) u[i] = feeder ? 0.f : coef[size_t(tIdx) * 12 + i];
  const int P = C > 136 ? C : 136;
  const int nB = P >> 2, cBlocks = C >> 2;
  const int nGroups = (R - 2 + 29) / 30;
  const int nIter = nGroups * nB + 31;
  const int64_t wrapStep = 30 * t.pitch - 4 * int64_t(nB);  // block nB of row r -> block 0 of row r+30
  float av[8], bv[8];  // rows r-1 / r-2 as float, columns c0-2 .. c0+5
#pragma unroll
  for (int i = 0; i < 8; i++) { av[i] = 0.f; bv[i] = 0.f; }
  float f1 = 0.f, f2 = 0.f;           // own row, columns c-1 and c-2
  float pf0 = 0.f, pf1 = 0.f;         // own outputs 0,1 of the previous block as float (columns 0,1 for the lane below)
  int32_t h1 = 0;                     // own row, column c-1 (integer, for the two Triangle columns)
  int32_t po1 = 0, po2 = 0, po3 = 0;  // own outputs of the previous block (Triangle operands of the lane below)
  int cb = -lane, r = lane;
  int32_t* p = t.base + int64_t(r) * t.pitch + 4 * cb;  // block cb of row r; dereferenced only while in range
  // The block's four cells (residuals; final values for the feeders and in columns 0,1) are fetched ONE ITERATION AHEAD.
  // Plain loads are enough for the feeders: the rows they read were stored by lanes of this same warp at least two
  // iterations earlier, and the __syncwarp that ends every iteration orders memory among the warp's lanes.
  int4 vN = make_int4(0, 0, 0, 0);
  if (cb == 0 && r < R) vN = *reinterpret_cast<const int4*>(p);
  for (int it = 0; it < nIter; it++) {
    const bool act = cb >= 0 && cb < cBlocks && r < R;
    const bool first = cb == 0;
    const bool triangle = cb == cBlocks - 1 && !feeder;
    const int4 v = vN;
    int32_t* const cur = p;
    cb++;
    p += 4;
    if (cb == nB) { cb = 0; r += 30; p += wrapStep; }
    if (cb >= 0 && cb < cBlocks && r < R) vN = *reinterpret_cast<const int4*>(p);
    // once-per-row operands, taken from the lane above BEFORE the windows shift (it finished its block 0 last iteration)
    const float s0 = __shfl_up_sync(0xffffffffu, pf0, 1);
    const float s1 = __shfl_up_sync(0xffffffffu, pf1, 1);
    const float s2 = __shfl_up_sync(0xffffffffu, av[2], 1);
    const float s3 = __shfl_up_sync(0xffffffffu, av[3], 1);
#pragma unroll
    for (int i = 0; i < 4; i++) { av[i] = av[i + 4]; bv[i] = bv[i + 4]; }
    if (first) { av[2] = s0; av[3] = s1; bv[2] = s2; bv[3] = s3; }
    // Triangle columns: row r-1, columns C-3..C-1 = lane l-1's outputs of its previous (= its last) block
    const int32_t upy = __shfl_up_sync(0xffffffffu, po1, 1);
    const int32_t upz = __shfl_up_sync(0xffffffffu, po2, 1);
    const int32_t upw = __shfl_up_sync(0xffffffffu, po3, 1);
    int32_t out[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      av[4 + j] = __shfl_up_sync(0xffffffffu, f2, 1);
      bv[4 + j] = __shfl_up_sync(0xffffffffu, av[j], 1);
      const int32_t res = j == 0 ? v.x : j == 1 ? v.y : j == 2 ? v.z : v.w;
      // LsDecoder12.java:424-438 -- evaluated left to right in float32, no fused multiply-add.  Computed for every
      // column and discarded (select, no branch) for columns 0,1 and the two Triangle columns.
      float q = u[0] * f1;
      q = q + u[1] * av[j + 1];
      q = q + u[2] * av[j + 2];
      q = q + u[3] * av[j + 3];
      q = q + u[4] * av[j + 4];
      q = q + u[5] * f2;
      q = q + u[6] * av[j];
      q = q + u[7] * bv[j];
      q = q + u[8] * bv[j + 1];
      q = q + u[9] * bv[j + 2];
      q = q + u[10] * bv[j + 3];
      q = q + u[11] * bv[j + 4];
      uint32_t add = uint32_t(java_round(q));
      if (j < 2) {
        if (first) add = 0u;  // columns 0,1 hold their final values already
      } else {
        // last two columns: Triangle predictor (LsDecoder12.java:459-468); tile_cols % 4 == 0 puts them at j = 2,3
        const int32_t upc = j == 2 ? upz : upw, upl = j == 2 ? upy : upz;
        if (triangle) add = (uint32_t(h1) + uint32_t(upc)) - uint32_t(upl);
      }
      const int32_t val = int32_t(uint32_t(res) + add);
      out[j] = val;
      h1 = val;
      f2 = f1;
      f1 = float(val);
      if (j == 0) pf0 = f1;
      if (j == 1) pf1 = f1;
    }
    if (act && !feeder) *reinterpret_cast<int4*>(cur) = make_int4(out[0], out[1], out[2], out[3]);
    po1 = out[1]; po2 = out[2]; po3 = out[3];
    __syncwarp();
  }
}

// =====================================================================================================
// Encode (LsEncoder12.encode :122-219 with the canonical-Huffman body; LsOptimalPredictor12.encode :109-292)
// =====================================================================================================
namespace {

constexpr int kMomentQuantities = 104;  // 13 sums + 91 products (upper triangle incl. diagonal)
constexpr int kMomentPerRole = 26;

// quantity q: q < 13 -> z[q]; otherwise the (i,j) product with i <= j in row-major order of the upper triangle
__host__ __device__ constexpr int moment_i(int q) {
  int k = q - 13, i = 0;
  while (k >= 13 - i) { k -= 13 - i; i++; }
  return i;
}
__host__ __device__ constexpr int moment_j(int q) {
  int k = q - 13, i = 0;
  while (k >= 13 - i) { k -= 13 - i; i++; }
  return i + k;
}

// One accumulated quantity with COMPILE-TIME indices: `constexpr int i = moment_i(Q)` forces the index arithmetic out
// of the kernel, and z[] stays in registers (a run-time index would send it to local memory).
template <int Q>
__device__ __forceinline__ double moment_term(const double (&z)[13]) {
  if constexpr (Q < 13) return z[Q];
  else {
    constexpr int i = moment_i(Q), j = moment_j(Q);
    return z[i] * z[j];
  }
}
template <int ROLE, int... A>
__device__ __forceinline__ void moment_accumulate_seq(const double (&z)[13], double (&acc)[kMomentPerRole], std::integer_sequence<int, A...>) {
  ((acc[A] += moment_term<A * 4 + ROLE>(z)), ...);
}
template <int ROLE>
__device__ __forceinline__ void moment_accumulate(const double (&z)[13], double (&acc)[kMomentPerRole]) {
  moment_accumulate_seq<ROLE>(z, acc, std::make_integer_sequence<int, kMomentPerRole>{});
}

// Header bytes of the canonical-Huffman packing: 55, or 59 with the value checksum behind the coefficients.
__device__ __forceinline__ uint32_t lsop_canon_header_bytes(const EncodeArgs& a) { return a.valueCrc ? 59u : 55u; }

struct LsopEncShared {
  CanonEncShared E;
  BitWindow W;
  double part[kWarps][kMomentPerRole];
  double sums[kMomentQuantities];
  double M[13][13];
  double rhs[13];
  float u[12];
  int singular;
};

// JAMA LUDecomposition ctor + solve (util/jama/LUDecomposition.java:70-135, :253-286), one thread, FP64,
// identical operation order (compiled with -fmad=false).
__device__ bool lu_solve13(double (*LU)[13], double* X) {
  const int n = 13;
  int piv[13];
  for (int i = 0; i < n; i++) piv[i] = i;
  double col[13];
  for (int j = 0; j < n; j++) {
    for (int i = 0; i < n; i++) col[i] = LU[i][j];
    for (int i = 0; i < n; i++) {
      int kmax = i < j ? i : j;
      double s = 0.0;
      for (int k = 0; k < kmax; k++) s += LU[i][k] * col[k];
      col[i] -= s;
      LU[i][j] = col[i];
    }
    int p = j;
    for (int i = j + 1; i < n; i++)
      if (fabs(col[i]) > fabs(col[p])) p = i;
    if (p != j) {
      for (int k = 0; k < n; k++) { double t = LU[p][k]; LU[p][k] = LU[j][k]; LU[j][k] = t; }
      int k = piv[p]; piv[p] = piv[j]; piv[j] = k;
    }
    if (LU[j][j] != 0.0)
      for (int i = j + 1; i < n; i++) LU[i][j] /= LU[j][j];
  }
  for (int j = 0; j < n; j++)
    if (LU[j][j] == 0.0) return false;
  double B[13];
  for (int i = 0; i < n; i++) B[i] = X[piv[i]];
  for (int i = 0; i < n; i++) X[i] = B[i];
  for (int k = 0; k < n; k++)
    for (int i = k + 1; i < n; i++) X[i] -= X[k] * LU[i][k];
  for (int k = n - 1; k >= 0; k--) {
    X[k] /= LU[k][k];
    for (int i = 0; i < k; i++) X[i] -= X[k] * LU[i][k];
  }
  return true;
}

struct LsInitGet {  // initializer residuals in stream order (LsOptimalPredictor12.java:143-209)
  TileView t;
  __device__ __forceinline__ int32_t operator()(uint32_t k) const {
    int r, c;
    stream_to_cell(kStreamLsopInit, int(k), t.R, t.C, &r, &c);
    return residual_at(G4_PRED_TRIANGLE, t, r, c);  // row 0 / column 0 degrade to plain differences
  }
};

struct LsInteriorGet {  // interior residuals (LsOptimalPredictor12.java:254-282)
  TileView t;
  const float* u;
  __device__ __forceinline__ int32_t operator()(uint32_t k) const {
    const int w = t.C - 4;
    int rr = int(k) / w;
    int r = 2 + rr, c = 2 + int(k) - rr * w;
    const int32_t* row = t.row(r);
    const int32_t* up1 = row - t.pitch;
    const int32_t* up2 = up1 - t.pitch;
    float p = u[0] * float(row[c - 1]);
    p = p + u[1] * float(up1[c - 1]);
    p = p + u[2] * float(up1[c]);
    p = p + u[3] * float(up1[c + 1]);
    p = p + u[4] * float(up1[c + 2]);
    p = p + u[5] * float(row[c - 2]);
    p = p + u[6] * float(up1[c - 2]);
    p = p + u[7] * float(up2[c - 2]);
    p = p + u[8] * float(up2[c - 1]);
    p = p + u[9] * float(up2[c]);
    p = p + u[10] * float(up2[c + 1]);
    p = p + u[11] * float(up2[c + 2]);
    return int32_t(uint32_t(row[c]) - uint32_t(java_round(p)));
  }
};

}  // namespace

__global__ void __launch_bounds__(kThreads) lsop_encode_kernel(EncodeArgs a) {
  extern __shared__ __align__(16) unsigned char smemRaw[];
  LsopEncShared& S = *reinterpret_cast<LsopEncShared*>(smemRaw);
  __shared__ int sTile;
  __shared__ uint32_t sMaxAbs;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  uint8_t* pm = a.scratch + size_t(blockIdx.x) * a.scratchStride;
  for (;;) {
    __syncthreads();
    if (tid == 0) sTile = atomicAdd(a.counter, 1);
    __syncthreads();
    const int tIdx = sTile;
    if (tIdx >= nTiles) break;
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int R = t.R, C = t.C;
    uint32_t* outWords = reinterpret_cast<uint32_t*>(a.slots + size_t(tIdx) * a.slotBytes);
    const uint32_t capWords = uint32_t(a.slotBytes / 4);
    if (R < 6 || C < 6) {  // LsOptimalPredictor12.java:114-116
      if (tid == 0) { a.lens[tIdx] = 0; a.preds[tIdx] = 0; a.status[tIdx] = G4_DECLINED; }
      continue;
    }
    // ---- normal equations: s[i] += z[i], c[i][j] += z[i]*z[j] over the interior cells (:319-344) --------
    {
      const int role = warp & 3, group = warp >> 2;
      const int w = C - 4;
      const int nInterior = (R - 2) * w;
      // largest sample magnitude of the tile: decides below whether the partitioned sums are exact
      if (tid == 0) sMaxAbs = 0u;
      __syncthreads();
      {
        uint32_t mx = 0u;
        for (int m = tid; m < R * C; m += kThreads) {
          const int rr = m / C;
          const int32_t v = t.row(rr)[m - rr * C];
          const uint32_t av = v < 0 ? 0u - uint32_t(v) : uint32_t(v);
          mx = mx > av ? mx : av;
        }
        mx = __reduce_max_sync(0xffffffffu, mx);
        if (lane == 0) atomicMax(&sMaxAbs, mx);
      }
      double acc[kMomentPerRole];
#pragma unroll
      for (int i = 0; i < kMomentPerRole; i++) acc[i] = 0.0;
      for (int m = group * 32 + lane; m < nInterior; m += 64) {
        int rr = m / w;
        int r = 2 + rr, c = 2 + m - rr * w;
        const int32_t* row = t.row(r);
        const int32_t* up1 = row - t.pitch;
        const int32_t* up2 = up1 - t.pitch;
        double z[13];
        z[0] = row[c]; z[1] = row[c - 1]; z[2] = up1[c - 1]; z[3] = up1[c]; z[4] = up1[c + 1]; z[5] = up1[c + 2];
        z[6] = row[c - 2]; z[7] = up1[c - 2]; z[8] = up2[c - 2]; z[9] = up2[c - 1]; z[10] = up2[c]; z[11] = up2[c + 1];
        z[12] = up2[c + 2];
        switch (role) {
          case 0: moment_accumulate<0>(z, acc); break;
          case 1: moment_accumulate<1>(z, acc); break;
          case 2: moment_accumulate<2>(z, acc); break;
          default: moment_accumulate<3>(z, acc); break;
        }
      }
#pragma unroll
      for (int i = 0; i < kMomentPerRole; i++) {
        double v = acc[i];
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        if (lane == 0) S.part[warp][i] = v;
      }
      __syncthreads();
      if (tid < kMomentQuantities) S.sums[tid] = S.part[tid & 3][tid >> 2] + S.part[(tid & 3) + 4][tid >> 2];
      // The partition above adds in another order than the reference's single loop.  That is the same number as long as
      // every partial sum is an exactly representable integer: nInterior * max|z|^2 < 2^53 (terrain: about 2^42).
      // Otherwise (full-range samples) each quantity is re-accumulated by one thread in the reference's cell order.
      const double mag = double(sMaxAbs);
      if (!(double(nInterior) * mag * mag < 9007199254740992.0) && tid < kMomentQuantities) {
        const int dr[13] = {0, 0, -1, -1, -1, -1, 0, -1, -2, -2, -2, -2, -2};
        const int dc[13] = {0, -1, -1, 0, 1, 2, -2, -2, -2, -1, 0, 1, 2};
        const int qi = tid < 13 ? tid : moment_i(tid), qj = tid < 13 ? -1 : moment_j(tid);
        double accq = 0.0;
        for (int r = 2; r < R; r++) {
          const int32_t* ri = t.row(r + dr[qi]) + dc[qi];
          const int32_t* rj = qj >= 0 ? t.row(r + dr[qj]) + dc[qj] : ri;
          if (qj < 0) for (int c = 2; c < C - 2; c++) accq += double(ri[c]);
          else for (int c = 2; c < C - 2; c++) accq += double(ri[c]) * double(rj[c]);
        }
        S.sums[tid] = accq;
      }
      __syncthreads();
    }
    if (tid == 0) {
      // design matrix (:346-368): 12x12 moment block bordered by the sums (Lagrange constraint)
      double cfull[13][13];
      for (int q = 13; q < kMomentQuantities; q++) {
        int i = moment_i(q), j = moment_j(q);
        cfull[i][j] = S.sums[q];
        cfull[j][i] = S.sums[q];
      }
      for (int i = 0; i < 13; i++) for (int j = 0; j < 13; j++) S.M[i][j] = 0.0;
      for (int i = 1; i < 13; i++) {
        for (int j = 1; j < 13; j++) S.M[i - 1][j - 1] = cfull[i][j];
        S.M[i - 1][12] = S.sums[i];
      }
      for (int j = 1; j < 13; j++) S.M[12][j - 1] = S.sums[j];
      for (int i = 1; i < 13; i++) S.rhs[i - 1] = cfull[0][i];
      S.rhs[12] = S.sums[0];
      bool ok = lu_solve13(S.M, S.rhs);
      S.singular = ok ? 0 : 1;
      if (ok)
        for (int i = 0; i < 12; i++) S.u[i] = __double2float_rn(S.rhs[i]);
    }
    __syncthreads();
    if (S.singular) {  // RuntimeException("Matrix is singular.") -> null (:377-381)
      if (tid == 0) { a.lens[tIdx] = 0; a.preds[tIdx] = 0; a.status[tIdx] = G4_DECLINED; }
      continue;
    }
    // ---- packing: revised header (LsHeader.java:210-265) + two canonical streams in one bit store --------
    const uint32_t nInit = uint32_t(4 * R + 2 * C - 9);
    const uint32_t nInterior = uint32_t(R - 2) * uint32_t(C - 4);
    BitOut o;
    bitwin_reset(S.W, o, outWords, capWords);
    if (tid == 0) {
      WinSink sink{S.W.win, 0};
      sink.put(uint32_t(a.codecIndex) & 0xffu, 8);
      sink.put((a.valueCrc ? 0x80u : 0u) | 0x40u | 2u, 8);  // checksum flag | revision flag | COMPRESSION_TYPE_CANON_HUFFMAN
      sink.put(12, 8);
      sink.put(uint32_t(t.at(0, 0)), 32);
      for (int i = 0; i < 12; i++) sink.put(__float_as_uint(S.u[i]), 32);
      if (a.valueCrc) sink.put(a.valueCrc[tIdx], 32);
    }
    o.bitPos = lsop_canon_header_bytes(a) * 8u;
    __syncthreads();
    LsInitGet g1{t};
    LsInteriorGet g2{t, S.u};
    bool bad = false;
    bool clean = canon_histogram(S.E, g1, nInit);
    canon_build_code(S.E, pm);
    if (!clean && !canon_reconcile_escapes(S.E, g1, nInit)) bad = true;  // see g4_canon_enc.cuh
    else {
      canon_emit_stream(S.E, S.W, o, g1, nInit);
      clean = canon_histogram(S.E, g2, nInterior);
      canon_build_code(S.E, pm);
      if (!clean && !canon_reconcile_escapes(S.E, g2, nInterior)) bad = true;
      else canon_emit_stream(S.E, S.W, o, g2, nInterior);
    }
    if (bad) {
      if (tid == 0) { a.lens[tIdx] = 0; a.preds[tIdx] = 0; a.status[tIdx] = G4_DECLINED; }
      continue;
    }
    bitwin_finish(S.W, o);
    if (tid == 0) {
      uint32_t len = (o.bitPos + 7) >> 3;
      a.lens[tIdx] = len;
      a.preds[tIdx] = 2;  // compression type: canonical Huffman
      a.status[tIdx] = len <= a.slotBytes ? G4_OK : G4_ERR_CAPACITY;
    }
  }
}

// ---- Deflate alternative (LsEncoder12.java:170-218) ---------------------------------------------------------------
// After lsop_encode_kernel has written the canonical-Huffman packing (type 2) into the tile's slot, the initializer
// and interior residuals are M32 coded (LsOptimalPredictor12.java:143-282 fills both the int and the M32 forms),
// deflated at level 6 by the stream workers, and the packing is replaced by the type-1 form when
// insideN < canonLength and initN + insideN < canonLength (the reference compares bodies only, headers excluded).
namespace {
// The coefficients sit at bytes 7..54 of both header forms; only what follows them depends on the value checksum.
__device__ __forceinline__ void load_slot_coefficients(const uint8_t* slot, float* u) {
  if (threadIdx.x < 12) u[threadIdx.x] = __uint_as_float(load_le32(slot + 7 + 4 * threadIdx.x));
  __syncthreads();
}
}  // namespace

__global__ void __launch_bounds__(kThreads) lsop_m32_size_kernel(EncodeArgs a, uint32_t* inLen) {
  __shared__ uint32_t scan[kWarps + 1];
  __shared__ float u[12];
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (int tIdx = blockIdx.x; tIdx < nTiles; tIdx += gridDim.x) {
    __syncthreads();
    if (a.status[tIdx] != G4_OK || a.lens[tIdx] < lsop_canon_header_bytes(a)) {  // declined (too small / singular): nothing to deflate
      if (threadIdx.x == 0) inLen[2 * tIdx] = inLen[2 * tIdx + 1] = 0;
      continue;
    }
    const TileView t = tile_view(a.band, a.grid, tIdx);
    load_slot_coefficients(a.slots + size_t(tIdx) * a.slotBytes, u);
    const uint32_t nInit = uint32_t(4 * t.R + 2 * t.C - 9);
    const uint32_t nInterior = uint32_t(t.R - 2) * uint32_t(t.C - 4);
    uint32_t s0 = m32_stream_size(LsInitGet{t}, nInit, scan);
    uint32_t s1 = m32_stream_size(LsInteriorGet{t, u}, nInterior, scan);
    if (threadIdx.x == 0) { inLen[2 * tIdx] = s0; inLen[2 * tIdx + 1] = s1; }
  }
}

__global__ void __launch_bounds__(kThreads) lsop_m32_write_kernel(EncodeArgs a, const uint32_t* inLen, const uint64_t* inOff,
                                                                  uint8_t* inBuf) {
  __shared__ uint32_t scan[kWarps + 1];
  __shared__ float u[12];
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (int tIdx = blockIdx.x; tIdx < nTiles; tIdx += gridDim.x) {
    __syncthreads();
    if (inLen[2 * tIdx + 1] == 0) continue;
    const TileView t = tile_view(a.band, a.grid, tIdx);
    load_slot_coefficients(a.slots + size_t(tIdx) * a.slotBytes, u);
    const uint32_t nInit = uint32_t(4 * t.R + 2 * t.C - 9);
    const uint32_t nInterior = uint32_t(t.R - 2) * uint32_t(t.C - 4);
    uint8_t* d0 = inBuf + inOff[2 * tIdx];
    uint8_t* d1 = inBuf + inOff[2 * tIdx + 1];
    uint32_t w0 = m32_stream_write(LsInitGet{t}, nInit, d0, scan);
    uint32_t w1 = m32_stream_write(LsInteriorGet{t, u}, nInterior, d1, scan);
    if (threadIdx.x < 16) { d0[w0 + threadIdx.x] = 0; d1[w1 + threadIdx.x] = 0; }
  }
}

__global__ void __launch_bounds__(kThreads) lsop_pick_kernel(EncodeArgs a, const uint32_t* inLen, const uint64_t* inOff,
                                                             const uint8_t* outBuf, const uint32_t* outLen) {
  const int tid = threadIdx.x;
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (int tIdx = blockIdx.x; tIdx < nTiles; tIdx += gridDim.x) {
    if (inLen[2 * tIdx + 1] == 0) continue;
    const uint32_t canonLength = a.lens[tIdx] - lsop_canon_header_bytes(a);  // bodies only (Appendix C quirk 11)
    const uint32_t initN = outLen[2 * tIdx], insideN = outLen[2 * tIdx + 1];
    if (insideN == 0 || insideN >= canonLength) continue;         // LsEncoder12.java:185-190
    if (initN == 0 || initN + insideN >= canonLength) continue;   // :197-201
    const uint32_t body = lsop_canon_header_bytes(a) + 8u;       // [nInit][nInterior] then the checksum, if any
    const uint32_t len = body + initN + insideN;
    if (len > a.slotBytes) {
      if (tid == 0) a.status[tIdx] = G4_ERR_CAPACITY;
      continue;
    }
    uint8_t* slot = a.slots + size_t(tIdx) * a.slotBytes;
    if (tid == 0) {
      slot[1] = uint8_t((a.valueCrc ? 0x80u : 0u) | 0x40u | 1u);  // checksum flag | revision flag | COMPRESSION_TYPE_DEFLATE (LsHeader.java:220-245)
      const uint32_t n0 = inLen[2 * tIdx], n1 = inLen[2 * tIdx + 1];
      for (int k = 0; k < 4; k++) { slot[55 + k] = uint8_t(n0 >> (8 * k)); slot[59 + k] = uint8_t(n1 >> (8 * k)); }
      if (a.valueCrc)
        for (int k = 0; k < 4; k++) slot[63 + k] = uint8_t(a.valueCrc[tIdx] >> (8 * k));
      a.lens[tIdx] = len;
      a.preds[tIdx] = 1;
    }
    const uint8_t* s0 = outBuf + inOff[2 * tIdx] + 112ull * uint64_t(2 * tIdx);
    const uint8_t* s1 = outBuf + inOff[2 * tIdx + 1] + 112ull * uint64_t(2 * tIdx + 1);
    for (uint32_t i = tid; i < initN; i += kThreads) slot[body + i] = s0[i];
    for (uint32_t i = tid; i < insideN; i += kThreads) slot[body + initN + i] = s1[i];
  }
}

cudaError_t launch_lsop_m32_size(const EncodeArgs& a, uint32_t* inLen, int nCtas, cudaStream_t s) {
  lsop_m32_size_kernel<<<nCtas, kThreads, 0, s>>>(a, inLen);
  return cudaGetLastError();
}
cudaError_t launch_lsop_m32_write(const EncodeArgs& a, const uint32_t* inLen, const uint64_t* inOff, uint8_t* inBuf, int nCtas,
                                  cudaStream_t s) {
  lsop_m32_write_kernel<<<nCtas, kThreads, 0, s>>>(a, inLen, inOff, inBuf);
  return cudaGetLastError();
}
cudaError_t launch_lsop_pick(const EncodeArgs& a, const uint32_t* inLen, const uint64_t* inOff, const uint8_t* outBuf,
                             const uint32_t* outLen, int nCtas, cudaStream_t s) {
  lsop_pick_kernel<<<nCtas, kThreads, 0, s>>>(a, inLen, inOff, outBuf, outLen);
  return cudaGetLastError();
}

cudaError_t launch_lsop_encode(const EncodeArgs& a, int nCtas, cudaStream_t s) {
  static std::atomic<uint64_t> attr{0};
  cudaError_t ea = once_per_device(attr, [] {
    return cudaFuncSetAttribute(lsop_encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(LsopEncShared)));
  });
  if (ea != cudaSuccess) return ea;
  lsop_encode_kernel<<<nCtas, kThreads, sizeof(LsopEncShared), s>>>(a);
  return cudaGetLastError();
}

size_t lsop_meta_bytes() { return kLsopMetaBytes; }

cudaError_t launch_lsop08_decode(const DecodeArgs& a, float* coef, int nCtas, int nTilesUpper, cudaStream_t s) {
  lsop08_decode_entropy_kernel<<<nCtas < 296 ? nCtas : 296, kThreads, 0, s>>>(a, coef);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  lsop08_wavefront_kernel<<<(nTilesUpper + kWarps - 1) / kWarps, kThreads, 0, s>>>(a, coef);
  return cudaGetLastError();
}

cudaError_t launch_lsop_decode(const DecodeArgs& a, float* coef, uint8_t* meta, int* defer, int* deferCounters, int nCtas,
                               int nTilesUpper, cudaStream_t s, int* launches,
                               const LsopFastArgs* fast, int smCount) {
  if (fast) {
    // g4_lsop_fast.cu takes every canonical-Huffman tile; what it cannot take (legacy Huffman / Deflate bodies, oversized
    // packings, tiles outside the fast arithmetic's range) comes back in `defer` and goes through the general kernels
    LsopFastArgs A = *fast;
    A.a = a;
    A.coef = coef;
    A.meta = meta;
    A.defer = defer;
    A.deferCount = deferCounters;
    int nLaunch = 0;
    cudaError_t e = launch_lsop_decode_fast(A, nTilesUpper, smCount, deferCounters + 2, s, &nLaunch);
    if (e != cudaSuccess) return e;
    DecodeArgs d = a;
    d.list = defer;
    d.listCount = deferCounters;
    d.counter = deferCounters + 1;
    lsop_decode_entropy_kernel<<<nCtas < 296 ? nCtas : 296, kThreads, 0, s>>>(d, coef);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    lsop_wavefront_kernel<<<(nTilesUpper + kWarps - 1) / kWarps, kThreads, 0, s>>>(d, coef);
    if (launches) *launches = nLaunch + 2;
    return cudaGetLastError();
  }
  // Staging capacity of the text kernel: 5 bits per sample of the tile, at least the default 28 KB (four CTAs per SM; 5.3
  // bits per sample of a 180x240 tile), at most what leaves one CTA per SM; packings beyond it go to the general kernels.
  constexpr uint32_t kMaxStageWords = (192u * 1024u) / 4u;
  uint32_t stageWords = uint32_t((uint64_t(a.band.tile_rows) * uint64_t(a.band.tile_cols) * 5 / 8 + 3) / 4);
  if (stageWords < uint32_t(kFastStageWords)) stageWords = kFastStageWords;
  if (stageWords > kMaxStageWords) stageWords = kMaxStageWords;
  stageWords = (stageWords + 255u) & ~255u;
  const size_t textSmem = canon_fast_smem_bytes(stageWords);
  static std::atomic<uint64_t> attr{0};
  {
    cudaError_t ea = once_per_device(attr, [] {
      const int maxSmem = int(canon_fast_smem_bytes(kMaxStageWords));
      cudaError_t e1 = cudaFuncSetAttribute(lsop_decode_text_kernel<InteriorRunSink>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxSmem);
      if (e1 == cudaSuccess)
        e1 = cudaFuncSetAttribute(lsop_decode_text_kernel<InteriorPackedSink>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxSmem);
      return e1;
    });
    if (ea != cudaSuccess) return ea;
  }
  const bool aligned = (a.band.tile_cols % 4) == 0 && (a.band.grid_pitch % 4) == 0 && a.band.tile_cols >= 8 &&
                       (reinterpret_cast<uintptr_t>(a.grid) & 15) == 0;
  // deferCounters[0] = number of deferred tiles (filled by kernel H), [1] = work counter of the general kernel,
  // [2] = work counter of the text kernel
  const int nBlocks = (nTilesUpper + kWarps - 1) / kWarps;
  lsop_decode_head_kernel<<<nBlocks, kThreads, 0, s>>>(a, coef, meta, defer, deferCounters, stageWords);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  DecodeArgs t = a;
  t.counter = deferCounters + 2;
  const int ctas = nCtas < nTilesUpper ? nCtas : nTilesUpper;
  if (aligned) lsop_decode_text_kernel<InteriorPackedSink><<<ctas, kThreads, textSmem, s>>>(t, meta);
  else lsop_decode_text_kernel<InteriorRunSink><<<ctas, kThreads, textSmem, s>>>(t, meta);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  DecodeArgs d = a;
  d.list = defer;
  d.listCount = deferCounters;
  d.counter = deferCounters + 1;
  lsop_decode_entropy_kernel<<<nCtas < 296 ? nCtas : 296, kThreads, 0, s>>>(d, coef);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (aligned) lsop_wavefront4_kernel<<<nBlocks, kThreads, 0, s>>>(a, coef);
  else lsop_wavefront_kernel<<<nBlocks, kThreads, 0, s>>>(a, coef);
  if (launches) *launches = 4;
  return cudaGetLastError();
}

}  // namespace g4
