// g4_lsop_fast.cu -- LSOP12 decode, fast path for sm_100a: byte hand-over + TMA-fed wavefront.
//
// Reference (under /root/reference/core/src/main/java/org/gridfour/lsop/): LsDecoder12.java:94-470 (decode,
// unpackInitializers, unpackInterior), LsHeader.java:104-189; canonical Huffman text:
// compress/canonicalHuffman/CanonicalHuffman.java:441-519.
//
// Three kernels over the canonical-Huffman (type 2) LSOP tiles of a band whose rows are 16-byte aligned:
//   H  lsop2_head_kernel   one warp per tile.  LSOP header, both code tables, the initializer stream (about 4R+2C
//      values) decoded into SHARED memory, where all initializer scans run: rows 0 and 1 leave as whole coalesced
//      rows; for every other row a 16-byte side record {v[r][0], v[r][1], D2[r], D1[r]} is written, D2/D1 being the
//      column prefix sums that turn the Triangle predictor of the last two columns (LsDecoder12.java:459-468) into
//      v[r][C-2] = v[r][C-3] + D2[r], v[r][C-1] = v[r][C-2] + D1[r] -- no dependence on the row above is left.
//   T  lsop2_text_kernel   one 512-thread CTA per tile.  The packing is staged into shared memory by ONE bulk-async
//      copy (cp.async.bulk + mbarrier) while the tables and the multi-symbol LUT are built; the interior residuals
//      leave as ONE BYTE each (symbol = residual + 128) into a shared-memory image of the tile's residual scratch,
//      which goes to HBM with one bulk-async store.  Residuals that do not fit a byte (escapes, nulls) are written as
//      byte 0 plus an entry in a small per-tile exception list.
//   W  lsop3_wave_kernel   one warp per tile, or one 16-lane half-warp per tile when the tile's columns fit 16 strips
//      (LsopFastGeom::tilesPerWarp; the two tiles of a warp share only its instruction stream and ring: wider strips
//      give fewer ramp steps and spread the fixed cost of a step over more cells).  The causal 12-tap float32 stencil as
//      a wavefront over COLUMN STRIPS:
//      lane k owns the W columns 2 + k W .. (W = 4, 8 or 16), walks down the rows and is one ROW behind lane k - 1
//      (row r of strip k needs row r of strip k - 1 and rows r - 1, r - 2 of strip k + 1).  Every lane is at the same
//      cell of its strip at the same time, so the control flow is uniform: no per-lane row ends, no wrap blocks; the
//      first two columns enter lane 0 as its "left neighbour", the Triangle-predicted last two columns are two cells of
//      the last lane.  Per row a lane receives its two left values by shuffle-up, two right values of the row above
//      by shuffle-down, reads its W residual bytes with one shared-memory load and writes one aligned 4 W-byte
//      piece of the raster row {left2, left1, cells 0 .. W-3}.  The residual image is laid out by the text kernel
//      in STEP order (image row s = strip k of tile row s - k, for all k): a wavefront step reads nStrips * W
//      contiguous bytes, fetched 128 / W steps at a time by cp.async.bulk + mbarrier into a two-stage ring.
//
// Arithmetic of one cell (bit-identical to the reference for |p| < 2^21, checked per cell):
//   p   = u1*z1 + ... + u12*z12          strictly left to right, float32, no FMA (-fmad=false)
//   t1  = RD(p + 1.5*2^22)               multiples of 1/2: 1.5*2^22 + floor(2p)/2, exactly
//   t2  = RD(t1 + (1.5*2^22 + 0.5))      integers:         1.5*2^23 + floor(p + 1/2)  == StrictMath.round(p)
//   val = residual + (bits(t2) - bits(1.5*2^23))
//   float(val) = t2 + (float(residual) - 1.5*2^23)      exact, |val| < 2^24; the second operand does not depend on p
// which is 12 FMUL + 11 FADD + 3 FADD per cell on the dependent chain (the Java formula needs 23) and one integer add;
// the two round-down adds were verified against Math.round for every float32 in (-2^21, 2^21) (DESIGN.md).
// A tile that leaves that range (or holds too many exceptions) is handed to the general kernels of g4_lsop.cu.
#include <cuda.h>
#include <cstdio>
#include <type_traits>
#include "g4_kernels.h"
#include "g4_predict.cuh"
#include "g4_lsop_common.cuh"

namespace g4 {

namespace {

constexpr int kTextThreads = 512;              // text kernel: threads per CTA for tiles of more than kTextSmallTile samples
constexpr int kTextThreadsSmall = 256;         // ... and for smaller tiles (four CTAs per SM instead of two)
constexpr uint32_t kTextSmallTile = 16384;
constexpr uint32_t kTextSubBits = 320;        // target sub-sequence size of the text kernel: one sub-sequence per thread for a 180x240 tile
constexpr int kExcWords = 128;               // per tile: [0] count, [2+2i] interior index, [3+2i] value
constexpr int kExcCap = (kExcWords - 2) / 2;  // 63 exceptions; more -> general path
constexpr uint32_t kTextLookback = 96;        // first pass of the staged text decode: bits before a sub-sequence limit where it starts
constexpr int kStageWordsPerThread = 22;  // registers that carry a thread's staged symbol bytes across the barrier
constexpr int kSpillWords = 8;            // words behind every slot in a per-CTA global scratch (stays in L2): the slots hold only
                                          // about 7 % more than the average sub-sequence, so the longer ones spill their tail
constexpr int kResidGuard = 256;             // bytes in front of the first tile of the residual scratch
constexpr float kMagicHalf = 6291456.0f;     // 1.5 * 2^22
constexpr float kMagicHalfUp = 6291456.5f;   // 1.5 * 2^22 + 1/2
constexpr float kMagicInt = 12582912.0f;     // 1.5 * 2^23, bits 0x4B400000
constexpr float kRange = 2097152.0f;         // 2^21

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
// shared memory of the text kernel in front of the tile image: CanonFastShared with a staging array of stageWords (+ 8) words --
// its LAST member, so the struct may be allocated shorter or longer than its declared size
__host__ __device__ constexpr size_t text_fast_bytes(uint32_t stageWords) {
  return (offsetof(CanonFastShared, sw) + size_t(stageWords + 8u) * 4u + 127u) & ~size_t(127);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done)
                 : "r"(bar), "r"(parity)
                 : "memory");
}

// residual image shared by kernels T and W (LsopFastGeom in g4_kernels.h): interior cell (row r, column c), r >= 2,
// 2 <= c < C - 2, has data column p = c - 2 and lies in strip p / W; wavefront step s = (r - 2) + p / W reads it, so its
// byte sits at image row s, byte p.  Data words (4 bytes, p a multiple of 4) never straddle a strip.
__device__ __forceinline__ uint32_t image_offset(uint32_t w, int logW, uint32_t P, uint32_t k) {  // w = C - 4
  const uint32_t rr = k / w, pp = k - rr * w;
  return (rr + (pp >> logW)) * P + pp;
}

// ---- kernel H -----------------------------------------------------------------------------------------------------
// p[i] <- carry + p[0] + ... + p[i] (mod 2^32), i < n; one warp, shared memory.  Returns the last value.
__device__ inline uint32_t warp_scan_inplace(int32_t* p, int n, uint32_t carry, int stride = 1) {
  const int lane = threadIdx.x & 31;
  for (int i0 = 0; i0 < n; i0 += 32) {
    const int i = i0 + lane;
    const uint32_t x = i < n ? uint32_t(p[i * stride]) : 0u;
    const uint32_t inc = warp_inclusive_scan(x);
    if (i < n) p[i * stride] = int32_t(carry + inc);
    carry += __shfl_sync(0xffffffffu, inc, 31);
  }
  __syncwarp();
  return carry;
}

__global__ void __launch_bounds__(kThreads, 3) lsop2_head_kernel(LsopFastArgs A, uint32_t maxPackBytes, int listBegin, int listEnd) {
  extern __shared__ __align__(16) unsigned char headSmem[];
  const DecodeArgs& a = A.a;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int R = A.g.R, C = A.g.C;
  const uint32_t nInit = uint32_t(4 * R + 2 * C - 9);
  const size_t perWarp = ((sizeof(CanonWarpShared) + 15) & ~size_t(15)) + ((size_t(nInit) * 4 + 15) & ~size_t(15));
  CanonWarpShared& W = *reinterpret_cast<CanonWarpShared*>(headSmem + perWarp * warp);
  int32_t* init = reinterpret_cast<int32_t*>(headSmem + perWarp * warp + ((sizeof(CanonWarpShared) + 15) & ~size_t(15)));
  const int li = listBegin + blockIdx.x * kWarps + warp;
  if (li >= listEnd || li >= *a.listCount) return;
  const int tIdx = a.list[li];
  uint8_t* m = A.meta + size_t(tIdx) * kLsopMetaBytes;
  if (lane == 0) {
    *reinterpret_cast<uint32_t*>(m) = 0;
    A.exc[size_t(tIdx) * kExcWords] = 0;
  }
  const TileView t = tile_view(a.band, a.grid, tIdx);
  const uint8_t* packing = a.arena + a.offsets[tIdx];
  const uint32_t len = a.lens[tIdx];
  LsHeaderInfo h = parse_ls_header(packing, len, A.coef + size_t(tIdx) * 12, lane == 0);
  if (lane == 0 && a.lsopCks && h.ok && h.hasChecksum) { a.lsopCks[2 * tIdx] = 1u; a.lsopCks[2 * tIdx + 1] = h.valueChecksum; }
  if (!h.ok) {
    if (lane == 0) a.status[tIdx] = G4_ERR_FORMAT;
    return;
  }
  if (h.type != 2 || len + 96u > maxPackBytes) {  // legacy Huffman / Deflate bodies, oversized packings: general kernels
    if (lane == 0) A.defer[atomicAdd(A.deferCount, 1)] = tIdx;
    return;
  }
  BitSrc src;
  src.init(packing, len);  // absolute bit positions inside the packing
  canon_warp_parse_header(W, src, h.headerSize * 8u);
  int status = W.error ? G4_ERR_FORMAT : G4_OK;
  uint32_t endBit = 0;
  if (status == G4_OK) {
    uint32_t eb = 0, nv = 0;
    auto emit = [&](uint32_t k, int32_t v) { init[k] = v; };
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
      for (int i = lane; i < kCanonSymbols; i += 32) {
        m[8 + i] = W.lens[i];
        reinterpret_cast<uint16_t*>(m + kLsopMetaSorted)[i] = W.sorted[i];
      }
      if (lane < 17) {  // the decoding tables, so that kernel T does not build them a second time
        reinterpret_cast<uint16_t*>(m + kLsopMetaFirst)[lane] = W.firstCode[lane];
        reinterpret_cast<uint16_t*>(m + kLsopMetaCount)[lane] = W.count[lane];
        reinterpret_cast<uint16_t*>(m + kLsopMetaOffset)[lane] = W.offset[lane];
      }
      if (lane == 0) *reinterpret_cast<uint32_t*>(m) = W.textStart;
    }
  }
  if (status == G4_OK) {
    // LsDecoder12.unpackInitializers (:204-241) on the stream-ordered values in shared memory
    int32_t* sA = init;                      // row 0, columns 1..C-1
    int32_t* sB = sA + (C - 1);              // column 0, rows 1..R-1
    int32_t* sC = sB + (R - 1);              // row 1, columns 1..C-1
    int32_t* sD = sC + (C - 1);              // column 1, rows 2..R-1
    int32_t* sE = sD + (R - 2);              // (r, C-2), (r, C-1) for r = 2..R-1
    const uint32_t seed = uint32_t(h.seed);
    warp_scan_inplace(sA, C - 1, seed);      // v[0][c]
    warp_scan_inplace(sB, R - 1, seed);      // v[r][0]
    // row 1: T[c] = v[1][c] - v[0][c], T[c] = T[c-1] + residual(1,c)
    warp_scan_inplace(sC, C - 1, uint32_t(sB[0]) - seed);
    for (int i = lane; i < C - 1; i += 32) sC[i] = int32_t(uint32_t(sC[i]) + uint32_t(sA[i]));  // v[1][c]
    __syncwarp();
    // column 1: U[r] = v[r][1] - v[r][0], U[r] = U[r-1] + residual(r,1)
    warp_scan_inplace(sD, R - 2, uint32_t(sC[0]) - uint32_t(sB[0]));
    // last two columns: D2[r] = v[r][C-2] - v[r][C-3] = D2[r-1] + residual(r,C-2); D1 the same one column further
    warp_scan_inplace(sE, R - 2, uint32_t(sC[C - 3]) - uint32_t(sC[C - 4]), 2);
    warp_scan_inplace(sE + 1, R - 2, uint32_t(sC[C - 2]) - uint32_t(sC[C - 3]), 2);
    int32_t* row0 = t.row(0);
    int32_t* row1 = t.row(1);
    for (int c = lane; c < C; c += 32) {
      row0[c] = c ? sA[c - 1] : int32_t(seed);
      row1[c] = c ? sC[c - 1] : sB[0];
    }
    int4* side = A.side + size_t(tIdx) * R;
    for (int r = lane; r < R; r += 32) {
      int4 s;
      if (r == 0) s = make_int4(int32_t(seed), sA[0], 0, 0);
      else if (r == 1) s = make_int4(sB[0], sC[0], 0, 0);
      else s = make_int4(sB[r - 1], int32_t(uint32_t(sB[r - 1]) + uint32_t(sD[r - 2])), sE[2 * (r - 2)], sE[2 * (r - 2) + 1]);
      side[r] = s;
    }
  }
  if (lane == 0) a.status[tIdx] = status;
}

// ---- kernel T -----------------------------------------------------------------------------------------------------
// Sink of the text decoder's packed write pass: one byte per value into the shared-memory image of the tile's residual
// scratch.  A run starts at any byte; its head goes out byte by byte up to the next word, the rest as aligned words
// (every row of the image is a whole number of words).
struct ByteTileSink {
  static constexpr bool kPacked = true;
  uint8_t* tile;       // shared memory, tileBytes
  uint32_t* exc;       // this tile's exception list (global)
  int w;               // C - 4, data bytes per row
  int logW;
  uint32_t P, Wm1;     // image row pitch, W - 1
  uint32_t addr;       // word-aligned image offset of queue byte 0
  uint32_t rowBase;    // image offset of data column 0 of the current row
  int left;            // data bytes from addr to the end of the row (a multiple of 4)
  int kAddr;           // interior index of the byte at addr
  int head;            // dummy bytes at the front of the queue (run head inside a word), 0 after the first store
  int cnt;             // queued bytes, dummies included; < 4 between calls
  uint64_t q;
  int excK, excSlot;   // the last exception this thread recorded
  int32_t excV;

  __device__ __forceinline__ void init(uint8_t* img, uint32_t* e, const LsopFastGeom& geom) {
    tile = img;
    exc = e;
    logW = geom.logW;
    w = geom.C - 4;
    P = uint32_t(geom.P);
    Wm1 = uint32_t(geom.W - 1);
  }
  __device__ __forceinline__ void begin(uint32_t k0) {
    const int rr = int(k0) / w, pp = int(k0) - rr * w;
    rowBase = uint32_t(rr) * P;
    const uint32_t a0 = rowBase + (uint32_t(pp) >> logW) * P + uint32_t(pp);
    head = pp & 3;
    addr = a0 & ~3u;
    left = w - (pp & ~3);
    kAddr = int(k0) - head;
    cnt = head;
    q = 0;
    excK = -1;
    excSlot = 0;
    excV = 0;
  }
  __device__ __forceinline__ int cur_k() const { return kAddr + cnt; }  // interior index of the value that will be queued next
  __device__ __forceinline__ void store_word() {  // cnt >= 4
    if (head) {
      for (int i = head; i < 4; i++) tile[addr + i] = uint8_t(q >> (8 * i));
      head = 0;
    } else *reinterpret_cast<uint32_t*>(tile + addr) = uint32_t(q);
    q >>= 32;
    cnt -= 4;
    kAddr += 4;
    step();
  }
  __device__ __forceinline__ void step() {  // on to the next word of the interior's row-major order
    addr += 4;
    left -= 4;
    if ((addr & Wm1) == 0u) {  // next strip: one image row further down; at the end of the row back to strip 0 of the next row
      addr += P;
      if (left == 0) {
        rowBase += P;
        addr = rowBase;
        left = w;
      }
    } else if (__builtin_expect(left == 0, 0)) {  // (a row that ends inside a strip)
      rowBase += P;
      addr = rowBase;
      left = w;
    }
  }
  // word copy of the staged form: bytes lo .. hi-1 of the destination word at addr are data (hi may exceed 4)
  __device__ __forceinline__ void put_word(uint32_t dw, int lo, int hi) {
    if (lo == 0 && hi >= 4) *reinterpret_cast<uint32_t*>(tile + addr) = dw;
    else
      for (int b = lo; b < hi && b < 4; b++) tile[addr + b] = uint8_t(dw >> (8 * b));
    step();
  }
  __device__ __forceinline__ void push(uint32_t bytes, int n) {  // n = 1..4 symbol bytes, first value in the low byte
    q |= uint64_t(bytes) << (8 * cnt);
    cnt += n;
    if (cnt >= 4) store_word();
  }
  __device__ __forceinline__ int add_exception(int k, int32_t v) {
    const uint32_t slot = atomicAdd(exc, 1u);
    if (slot < uint32_t(kExcCap)) {
      exc[2 + 2 * slot] = uint32_t(k);
      exc[3 + 2 * slot] = uint32_t(v);
    }
    excK = k;
    excV = v;
    excSlot = int(slot);
    return int(slot);
  }
  __device__ __forceinline__ void put_rare(int32_t v) {  // a value that is no byte (null)
    add_exception(cur_k(), v);
    push(0u, 1);
  }
  // an escape extends the value before it (CanonicalHuffman.java:495-504): v = (v << nb) | bits
  __device__ __forceinline__ void amend(int nb, uint32_t bits) {
    const int kp = cur_k() - 1;
    if (kp == excK) {
      excV = int32_t((uint32_t(excV) << nb) | bits);
      if (excSlot < kExcCap) exc[3 + 2 * excSlot] = uint32_t(excV);
      return;
    }
    uint32_t b;
    if (cnt > head) {  // still queued
      const int sh = 8 * (cnt - 1);
      b = uint32_t(q >> sh) & 0xffu;
      q &= ~(0xffull << sh);
    } else {  // already in the image
      // (cnt == head: with head != 0 nothing of this run was stored yet, which `have` in the caller excludes)
      const uint32_t o = image_offset(uint32_t(w), logW, P, uint32_t(kp));
      b = tile[o];
      tile[o] = 0;
    }
    add_exception(kp, int32_t(((b - 128u) << nb) | bits));
  }
  __device__ __forceinline__ void end() {
    for (int i = head; i < cnt; i++) tile[addr + i] = uint8_t(q >> (8 * i));
  }
};

// ---- staged text decode -------------------------------------------------------------------------------------------
// canon_fast_decode_text decodes every bit at least twice: once to COUNT the values of each sub-sequence (their output
// positions are a prefix sum of the counts) and once to write them.  Here the counting pass also keeps the symbol
// bytes it sees: every sub-sequence has a small slot in the tile image itself (the image is not written before the
// prefix sum is known, so it is free), and after the prefix sum each thread takes its slot into registers, the CTA
// synchronises, and the bytes go to their place in the image -- a copy instead of a second decode.  A sub-sequence that
// outgrows its slot (the slots hold about 10 % more than the average) is decoded a second time like before; one that
// holds a value that is no byte (escape, null) is walked once more by text_exceptions_sub for the exception list.
constexpr int kSubRare = 4;      // S.eot[] flag: the sub-sequence holds an escape or a null
constexpr int kSubOverflow = 8;  // S.eot[] flag: more values than the slot holds

// Like canon_fast_count; additionally stores the symbol byte of every counted value to slot[0 .. slotWords) (shared memory).
// Bit window of the staging pass: two staged words and the absolute bit position (the funnel shift takes it modulo 32;
// a refill is due when a skip crosses a word boundary).
struct PosCursor {
  uint32_t lo, hi, next, pos;
  __device__ __forceinline__ void init(const uint32_t* sw, uint32_t p) {
    const uint32_t i = p >> 5;
    lo = sw[i];
    hi = sw[i + 1];
    next = i + 2;
    pos = p;
  }
  __device__ __forceinline__ uint32_t peek() const { return __funnelshift_r(lo, hi, pos); }
  __device__ __forceinline__ void skip(const uint32_t* sw, uint32_t n) {  // n <= 32
    const uint32_t np = pos + n;
    if ((np ^ pos) & 32u) {
      lo = hi;
      hi = sw[next++];
    }
    pos = np;
  }
};

// Byte accumulator of the staging pass: the pending (< 4) bytes sit TOP-justified in `acc`, so that they and the (up to
// three) symbol bytes of a lookup are contiguous in the pair (acc, m): the next output word is one funnel shift left, the
// new accumulator one funnel shift right -- no 64-bit queue.  qc8 = 8 x pending bytes.
struct ByteAcc {
  uint32_t acc, qc8, w;
  __device__ __forceinline__ void init() { acc = 0; qc8 = 0; w = 0; }
  // m24: symbol bytes in the low bytes (byte 3 zero), n8 = 8 x their number (8, 16 or 24)
  __device__ __forceinline__ void append(uint32_t m24, uint32_t n8, uint32_t* slot, uint32_t slotWords, uint32_t* spill) {
    const uint32_t out = __funnelshift_l(acc, m24, qc8);
    acc = __funnelshift_r(acc, m24, n8);
    qc8 += n8;
    if (qc8 >= 32u) {
      if (w < slotWords) slot[w] = out;
      else if (w - slotWords < uint32_t(kSpillWords)) spill[w - slotWords] = out;
      w++;
      qc8 -= 32u;
    }
  }
  __device__ __forceinline__ void finish(uint32_t* slot, uint32_t slotWords, uint32_t* spill) {
    if (qc8) {
      const uint32_t out = acc >> (32u - qc8);
      if (w < slotWords) slot[w] = out;
      else if (w - slotWords < uint32_t(kSpillWords)) spill[w - slotWords] = out;
      w++;
    }
  }
};

__device__ __forceinline__ void text_stage_sub(const CanonFastShared& S, uint32_t nBits, uint32_t start, uint32_t limit, uint32_t* slot,
                                               uint32_t slotWords, uint32_t* spill, uint32_t* endOut, uint32_t* cntOut, int* flagOut) {
  PosCursor cur;
  cur.init(S.sw, start);
  const int lastFull = int(limit) - kFastLutBits;  // the 11-bit window lies before the limit up to this position
  uint32_t c = 0, end;
  int flag = 0;
  ByteAcc A;
  A.init();
  for (;;) {
    if (int(cur.pos) <= lastFull) {
      const uint32_t m = S.mlut[cur.peek() & ((1u << kFastLutBits) - 1u)];
      const uint32_t n = m >> 28;
      if (n) {
        cur.skip(S.sw, (m >> 24) & 15u);
        c += n;
        A.append(m & 0xffffffu, (m >> 25) & 0x18u, slot, slotWords, spill);
        continue;
      }
    }
    const uint32_t e = S.lut[cur.peek() & ((1u << kFastLutBits) - 1u)];
    uint32_t byte;
    if (e - 1u < 0x7fffu) {  // LUT hit on a plain value: e = sym | len << 9
      if (cur.pos >= limit) { end = cur.pos; break; }
      cur.skip(S.sw, e >> 9);
      byte = e & 0xffu;
    } else {
      const uint32_t p0 = cur.pos;
      uint32_t after;
      const int sym = canon_fast_rare_symbol(S, e, p0, nBits, &after);
      if (sym < 0) { flag = 2; end = p0; break; }
      if (sym == kSymEsc2 || sym == kSymEsc8) {
        after += sym == kSymEsc2 ? 2u : 8u;
        if (after > nBits) { flag = 2; end = p0; break; }
        flag |= kSubRare;
        cur.init(S.sw, after);
        continue;
      }
      if (p0 >= limit) { end = p0; break; }
      if (sym == kSymEot) { flag |= 1; end = after; break; }
      if (sym == kSymNull) { flag |= kSubRare; byte = 0u; }
      else byte = uint32_t(sym);  // a byte value with a code longer than the LUT
      cur.init(S.sw, after);
    }
    c++;
    A.append(byte, 8u, slot, slotWords, spill);
  }
  A.finish(slot, slotWords, spill);
  if (A.w > slotWords + uint32_t(kSpillWords)) flag |= kSubOverflow;
  *endOut = end;
  *cntOut = c;
  *flagOut = flag;
}

// The write pass of canon_fast_decode_text for ONE sub-sequence (values from `start` up to the first value at or after
// `limit`), for the sub-sequences that did not fit their slot.  Returns false for a malformed stream.
__device__ __forceinline__ bool text_write_sub(const CanonFastShared& S, uint32_t nBits, uint32_t start, uint32_t limit, uint32_t k0,
                                            ByteTileSink& sink) {
  BitCursor cur;
  cur.init(S, start, limit);
  sink.begin(k0);
  bool have = false, ok = true;
  for (;;) {
    if (cur.rem >= kFastLutBits) {
      const uint32_t m = S.mlut[cur.peek() & ((1u << kFastLutBits) - 1u)];
      const uint32_t n = m >> 28;
      if (n) {
        cur.skip(S, (m >> 24) & 15u);
        sink.push(m & 0xffffffu, int(n));
        have = true;
        continue;
      }
    }
    const uint32_t e = S.lut[cur.peek() & ((1u << kFastLutBits) - 1u)];
    if (e - 1u < 0x7fffu) {  // plain value
      if (cur.rem <= 0) break;
      cur.skip(S, e >> 9);
      sink.push(e & 0xffu, 1);
      have = true;
      continue;
    }
    const uint32_t p0 = cur.pos(limit);
    uint32_t after;
    const int sym = canon_fast_rare_symbol(S, e, p0, nBits, &after);
    if (sym < 0) { ok = false; break; }
    if (sym == kSymEsc2 || sym == kSymEsc8) {
      const int nb = sym == kSymEsc2 ? 2 : 8;
      if (!have || after + nb > nBits) { ok = false; break; }
      SmemBitSrc src{S.sw, nBits};
      sink.amend(nb, src.bits(after, nb));
      after += nb;
    } else {
      if (p0 >= limit || sym == kSymEot) break;
      if (sym == kSymNull) sink.put_rare(INT32_MIN);
      else sink.push(uint32_t(sym), 1);  // a byte value with a code longer than the LUT
      have = true;
    }
    cur.init(S, after, limit);
  }
  sink.end();
  return ok;
}

// Exception-list entries of one sub-sequence whose values start at interior index k0 (the bytes are in the image).
__device__ __noinline__ void text_exceptions_sub(const CanonFastShared& S, uint32_t nBits, uint32_t start, uint32_t limit, uint32_t k0,
                                                 uint8_t* tile, uint32_t* exc, int w, int logW, uint32_t P) {
  auto image_off = [&](uint32_t k) { return image_offset(uint32_t(w), logW, P, k); };
  auto add = [&](uint32_t k, int32_t v) {
    const uint32_t slot = atomicAdd(exc, 1u);
    if (slot < uint32_t(kExcCap)) {
      exc[2 + 2 * slot] = k;
      exc[3 + 2 * slot] = uint32_t(v);
    }
  };
  SmemBitSrc src{S.sw, nBits};
  uint32_t pos = start, k = k0, pk = 0;
  bool pending = false;
  int32_t pv = 0;
  for (;;) {
    const uint32_t e = S.lut[src.peek32(pos) & ((1u << kFastLutBits) - 1u)];
    int sym;
    uint32_t after;
    if (e - 1u < 0x7fffu) { sym = int(e & 0xffu); after = pos + (e >> 9); }
    else {
      sym = canon_fast_rare_symbol(S, e, pos, nBits, &after);
      if (sym < 0) break;
    }
    if (sym == kSymEsc2 || sym == kSymEsc8) {  // extends the value before it (CanonicalHuffman.java:495-504): v = (v << nb) | bits
      const int nb = sym == kSymEsc2 ? 2 : 8;
      if (after + nb > nBits || k == k0) break;
      if (!pending) {
        pk = k - 1;
        const uint32_t o = image_off(pk);
        pv = int32_t(tile[o]) - 128;
        tile[o] = 0;
        pending = true;
      }
      pv = int32_t((uint32_t(pv) << nb) | src.bits(after, nb));
      after += nb;
    } else {
      if (pending) { add(pk, pv); pending = false; }
      if (pos >= limit || sym == kSymEot) break;
      if (sym == kSymNull) add(k, INT32_MIN);
      k++;
    }
    pos = after;
  }
  if (pending) add(pk, pv);
}

// Decodes the interior text (tables and LUT ready, text at bit T0) into the tile image.  All kTextThreads threads call.
// Returns 0 = done, 1 = malformed stream, 2 = the tile does not suit the staged form (caller uses canon_fast_decode_text).
template <int NT>
__device__ int lsop_text_decode(CanonFastShared& S, uint32_t nBits, const uint32_t T0, uint32_t nInterior, uint32_t imageBytes,
                                ByteTileSink sink, uint32_t* spillArea) {
  constexpr int kRounds = kFastMaxSub / NT;
  const int tid = threadIdx.x;
  const uint32_t avail = nBits - T0;
  uint32_t rounds = (avail / kTextSubBits + NT - 1) / NT;
  if (rounds < 1u) rounds = 1u;
  if (rounds > uint32_t(kRounds)) rounds = kRounds;
  uint32_t B = (avail + rounds * NT - 1) / (rounds * NT);
  if (B < 96u) B = 96u;
  const int nSub = int((avail + B - 1) / B);
  // slots: the image cut into nSub equal pieces, capped by what a thread can carry in registers
  uint32_t slotWords = (imageBytes / uint32_t(nSub)) >> 2;
  if (slotWords > uint32_t(kStageWordsPerThread) / rounds) slotWords = uint32_t(kStageWordsPerThread) / rounds;
  // not worth it unless slot + spill hold the average sub-sequence with room to spare (else most of them decode twice)
  if (uint64_t(slotWords + uint32_t(kSpillWords)) * 4u * uint64_t(nSub) * 3u < uint64_t(nInterior) * 4u) return 2;
  uint32_t* const image32 = reinterpret_cast<uint32_t*>(sink.tile);
  if (tid == 0) S.firstEot = nSub;
  // pass 0: only the END of every sub-sequence matters here, so start kTextLookback bits before the limit and rely on
  // self-synchronisation (sub-sequence 0 as well: every thread does the same amount)
#pragma unroll 1
  for (int i = tid; i < nSub; i += NT) {
    uint32_t limit = T0 + uint32_t(i + 1) * B;
    if (limit > nBits) limit = nBits;
    uint32_t from = T0 + uint32_t(i) * B;
    if (limit - from > kTextLookback) from = limit - kTextLookback;
    uint32_t e, c;
    int f;
    canon_fast_count(S, nBits, from, limit, &e, &c, &f);
    S.endpos[i] = e;
    S.startv[i] = 0xffffffffu;  // forces the exact decode of every sub-sequence in the first pass below
  }
  // synchronisation passes: sub-sequence i must start where i-1 ended (see canon_fast_decode_text)
  volatile uint32_t* vend = S.endpos;
  __syncthreads();
  for (int pass = 0; pass <= nSub; pass++) {
    bool any = false;
#pragma unroll 1
    for (int i = tid; i < nSub; i += NT) {
      const uint32_t ns = i ? vend[i - 1] : T0;
      if (ns != S.startv[i]) {
        S.startv[i] = ns;
        uint32_t limit = T0 + uint32_t(i + 1) * B;
        if (limit > nBits) limit = nBits;
        uint32_t e, c;
        int f;
        text_stage_sub(S, nBits, ns, limit, image32 + size_t(i) * slotWords, slotWords, spillArea + size_t(i) * kSpillWords, &e, &c, &f);
        vend[i] = e;
        S.cnt[i] = uint16_t(c);
        S.eot[i] = uint8_t(f);
        any = true;
      }
    }
    if (!__syncthreads_or(any ? 1 : 0)) break;
  }
#pragma unroll 1
  for (int i = tid; i < nSub; i += NT)
    if (S.eot[i] & 3) atomicMin(&S.firstEot, i);
  __syncthreads();
  const int fe = S.firstEot;
  if (fe == nSub || (S.eot[fe] & 3) == 2) return 1;  // no end-of-text, an invalid code, or the data ended early
  // value offsets: thread tid owns sub-sequences tid*kRounds .. +kRounds-1 for the scan
  uint32_t mySum = 0;
#pragma unroll
  for (int j = 0; j < kRounds; j++) {
    const int i = tid * kRounds + j;
    mySum += (i <= fe && i < nSub) ? S.cnt[i] : 0u;
  }
  uint32_t total;
  const uint32_t ex = block_exclusive_scan<NT>(mySum, S.scan, &total);
  if (total != nInterior) return 1;
  uint32_t* offv = S.endpos;  // end positions are no longer needed: the array now holds the first value index of every sub-sequence
  {
    uint32_t run = ex;
#pragma unroll
    for (int j = 0; j < kRounds; j++) {
      const int i = tid * kRounds + j;
      if (i < nSub) {
        offv[i] = run;
        run += (i <= fe) ? S.cnt[i] : 0u;
      }
    }
  }
  // slots -> registers (every thread: sub-sequences tid and tid + NT), barrier, registers -> their place in the image
  uint32_t r[kStageWordsPerThread];
#pragma unroll
  for (int j = 0; j < kStageWordsPerThread; j++) r[j] = 0;
  {
    const uint32_t perSub = uint32_t(kStageWordsPerThread) / rounds;
    for (uint32_t s = 0; s < rounds; s++) {
      const int i = tid + int(s) * NT;
      if (i <= fe && !(S.eot[i] & kSubOverflow)) {
        const uint32_t* slot = image32 + size_t(i) * slotWords;
#pragma unroll
        for (int j = 0; j < kStageWordsPerThread; j++)
          if (uint32_t(j) >= s * perSub && uint32_t(j) < s * perSub + slotWords) r[j] = slot[uint32_t(j) - s * perSub];
      }
    }
  }
  __syncthreads();
  bool bad = false;
  {
    const uint32_t perSub = uint32_t(kStageWordsPerThread) / rounds;
    for (uint32_t s = 0; s < rounds; s++) {
      const int i = tid + int(s) * NT;
      if (i > fe) continue;
      const uint32_t n = S.cnt[i];
      const int flags = S.eot[i];
      uint32_t limit = T0 + uint32_t(i + 1) * B;
      if (limit > nBits) limit = nBits;
      if (flags & kSubOverflow) {
        if (!text_write_sub(S, nBits, S.startv[i], limit, offv[i], sink)) bad = true;
        continue;
      }
      if (n == 0) continue;
      sink.begin(offv[i]);
      if (rounds == 1u) {
        // one sub-sequence per thread (the usual case): destination words are the source words funnel-shifted by the
        // run's byte offset inside its first word -- no byte queue; source word d = r[d], then the spilled tail
        const int head = sink.head;
        const uint32_t sh = 8u * uint32_t(head);
        const int nD = int((n + uint32_t(head) + 3u) >> 2);  // destination words touched
        const uint32_t* sp = spillArea + size_t(i) * kSpillWords;
        uint32_t prev = 0;
#pragma unroll
        for (int d = 0; d < kStageWordsPerThread + kSpillWords + 1; d++) {
          if (d >= nD) break;
          uint32_t cur = 0;
          if (d < kStageWordsPerThread && uint32_t(d) < slotWords) cur = r[d];
          else if (uint32_t(d) >= slotWords && uint32_t(d) - slotWords < uint32_t(kSpillWords) && 4u * uint32_t(d) < n) cur = sp[uint32_t(d) - slotWords];
          sink.put_word(__funnelshift_l(prev, cur, sh), d == 0 ? head : 0, int(n) + head - 4 * d);
          prev = cur;
        }
        if (flags & kSubRare) text_exceptions_sub(S, nBits, S.startv[i], limit, offv[i], sink.tile, sink.exc, sink.w, sink.logW, sink.P);
        continue;
      }
#pragma unroll
      for (int j = 0; j < kStageWordsPerThread; j++) {
        const uint32_t at = (uint32_t(j) - s * perSub) * 4u;  // byte position of word j inside this sub-sequence's slot
        if (uint32_t(j) >= s * perSub && uint32_t(j) < s * perSub + slotWords && at < n) {
          const uint32_t m = n - at;
          sink.push(m >= 4u ? r[j] : (r[j] & ((1u << (8 * m)) - 1u)), m >= 4u ? 4 : int(m));
        }
      }
      if (n > slotWords * 4u) {  // the tail this thread spilled in the staging pass
        const uint32_t* sp = spillArea + size_t(i) * kSpillWords;
        for (uint32_t at = slotWords * 4u; at < n; at += 4u) {
          const uint32_t wv = *sp++, m = n - at;
          sink.push(m >= 4u ? wv : (wv & ((1u << (8 * m)) - 1u)), m >= 4u ? 4 : int(m));
        }
      }
      sink.end();
      if (flags & kSubRare) text_exceptions_sub(S, nBits, S.startv[i], limit, offv[i], sink.tile, sink.exc, sink.w, sink.logW, sink.P);
    }
  }
  return __syncthreads_or(bad ? 1 : 0) ? 1 : 0;
}

template <int NT>
__global__ void __launch_bounds__(NT, NT == 512 ? 2 : 4) lsop2_text_kernel(LsopFastArgs A, uint32_t stageWords, int listBegin, int listEnd) {
  extern __shared__ __align__(128) unsigned char textSmem[];
  CanonFastShared& F = *reinterpret_cast<CanonFastShared*>(textSmem);
  uint8_t* tileImg = textSmem + text_fast_bytes(stageWords);
  __shared__ int sTile[2];
  __shared__ __align__(8) uint64_t sBar;
  const DecodeArgs& a = A.a;
  const int tid = threadIdx.x;
  const uint32_t bar = smem_u32(&sBar);
  if (tid == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;");
    sTile[0] = listBegin + atomicAdd(a.counter, 1);
  }
  __syncthreads();
  uint32_t parity = 0;
  for (int phase = 0;; phase ^= 1) {
    const int li = sTile[phase];
    if (li >= listEnd || li >= *a.listCount) break;
    // the tile after this one: fetched now, read after the barriers of this iteration
    if (tid == 0) sTile[phase ^ 1] = listBegin + atomicAdd(a.counter, 1);
    const int tIdx = a.list[li];
    const uint8_t* m = A.meta + size_t(tIdx) * kLsopMetaBytes;
    const uint32_t T0 = *reinterpret_cast<const uint32_t*>(m);
    if (T0 == 0) { __syncthreads(); continue; }  // deferred or rejected by kernel H
    const uint8_t* packing = a.arena + a.offsets[tIdx];
    const uint32_t len = a.lens[tIdx];
    // stage: the packing from its 16-byte line start; whole 16-byte pieces by ONE bulk-async copy, the tail by bytes
    const uint32_t delta = uint32_t(reinterpret_cast<uintptr_t>(packing) & 15u);
    const uint8_t* src16 = packing - delta;
    const uint32_t span = len + delta, nBulk = span & ~15u;
    if (tid == 0 && nBulk) {
      mbar_expect_tx(bar, nBulk);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(F.sw)), "l"(src16),
                   "r"(nBulk), "r"(bar)
                   : "memory");
    }
    if (tid < 64) {  // tail bytes and zero padding (the decoder reads whole words, up to 8 words past the data)
      const uint32_t i = nBulk + uint32_t(tid);
      reinterpret_cast<uint8_t*>(F.sw)[i] = i < span ? src16[i] : uint8_t(0);
    }
    // decoding tables as kernel H built (and validated) them
    for (int i = tid; i < kCanonSymbols; i += NT) F.sorted[i] = reinterpret_cast<const uint16_t*>(m + kLsopMetaSorted)[i];
    if (tid < 17) {
      F.firstCode[tid] = reinterpret_cast<const uint16_t*>(m + kLsopMetaFirst)[tid];
      F.count[tid] = reinterpret_cast<const uint16_t*>(m + kLsopMetaCount)[tid];
      F.offset[tid] = reinterpret_cast<const uint16_t*>(m + kLsopMetaOffset)[tid];
    }
    if (tid == 0) F.error = 0;
    __syncthreads();
    bool ok = true;
    canon_fast_build_lut<NT>(F);
    if (nBulk) mbar_wait(bar, parity);
    parity ^= nBulk ? 1u : 0u;
    __syncthreads();
    int rc = ok ? 0 : 1;
    if (ok) {
      const uint32_t nInterior = uint32_t(A.g.R - 2) * uint32_t(A.g.C - 4);
      ByteTileSink sink;
      sink.init(tileImg, A.exc + size_t(tIdx) * kExcWords, A.g);
      // the previous tile's image has left shared memory (a barrier follows before the image is written again)
      if (tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      rc = lsop_text_decode<NT>(F, span * 8u, T0 + 8u * delta, nInterior, uint32_t(A.g.tileBytes), sink,
                                reinterpret_cast<uint32_t*>(A.textStage) + size_t(blockIdx.x) * (kFastMaxSub * kSpillWords));
      if (rc == 2) {  // (uniform) the two-pass form
        uint32_t endBit = 0, nv = 0;
        rc = (canon_fast_decode_text<ByteTileSink, NT, kTextSubBits>(F, span * 8u, T0 + 8u * delta, nInterior, 0u, sink, &endBit, &nv) &&
              nv == nInterior) ? 0 : 1;
      }
      ok = rc == 0;
    }
    __syncthreads();
    if (tid == 0) {
      if (rc == 1) a.status[tIdx] = G4_ERR_FORMAT;
      else if (A.exc[size_t(tIdx) * kExcWords] > uint32_t(kExcCap)) {  // general kernels
        A.exc[size_t(tIdx) * kExcWords] = uint32_t(kExcCap) + 1u;                  // (the wavefront kernel skips the tile)
        A.defer[atomicAdd(A.deferCount, 1)] = tIdx;
      }
      else {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        uint8_t* dst = A.resid + kResidGuard + size_t(tIdx) * size_t(A.g.tilePitch);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(tileImg)), "r"(uint32_t(A.g.tileBytes))
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
  }
  if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- kernel W -----------------------------------------------------------------------------------------------------
#ifndef G4_WAVE_CTAS
#define G4_WAVE_CTAS 2
#endif
#ifndef G4_WAVE_WARPS
#define G4_WAVE_WARPS 8
#endif
constexpr int kWaveWarps = G4_WAVE_WARPS;  // warps (= tiles) per CTA of the wavefront kernel
constexpr int kWaveChunkBytes = 4096;  // ring stage: one bulk copy of 128 / W image rows (<= 32 strips x W bytes each)

// The value of an exceptional cell (byte 0 in the scratch): its list entry, or -128 when the byte was genuine.
// exc: the tile's list, which holds at most kExcCap entries (the wavefront skips tiles with more).
__device__ __noinline__ int32_t wave_exception(const uint32_t* exc, int k) {
  const int n = int(exc[0]);
  for (int i = 0; i < n; i++)
    if (int(exc[2 + 2 * i]) == k) return int32_t(exc[3 + 2 * i]);
  return -128;
}

// floats of rows 0 and 1 of the tile (written by kernel H), columns 0 .. C + 3 (zeros past C - 1), per tile of a warp
__device__ __forceinline__ int wave_rowbuf_floats(int C) { return (C + 4 + 3) & ~3; }

// PAIR: two tiles per warp (LsopFastGeom::tilesPerWarp), one per 16-lane half; lane & 15 is the strip, and the halves
// share nothing but the instruction stream and the warp's ring (each takes half of every stage).
template <int W, bool WIDE, bool PAIR>
__global__ void __launch_bounds__(32 * kWaveWarps, G4_WAVE_CTAS) lsop3_wave_kernel(LsopFastArgs A, int* tileCounter, int listBegin, int listEnd) {
  extern __shared__ __align__(128) unsigned char waveSmem[];
  constexpr int CR = 128 / W;   // image rows per chunk
  constexpr int NW = W / 4;     // residual words per lane and step
  constexpr int E = W - 4;      // the last strip: cells E, E + 1 are the row's last two columns (C a multiple of W)
  constexpr int TPW = PAIR ? 2 : 1;  // tiles per warp
  constexpr int HL = 32 / TPW;       // lanes per tile (the width of every shuffle)
  constexpr uint32_t kHalfStage = uint32_t(kWaveChunkBytes) / 2;
  // W 16 stores the first 8 columns of a strip row as soon as they are done: with the row's 14 outputs held to the end
  // of the step, pairs need more than 128 registers
  constexpr bool kEarlyLo = W == 16;
  const DecodeArgs& a = A.a;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int half = PAIR ? lane >> 4 : 0, ks = PAIR ? lane & 15 : lane;  // this lane's tile of the warp, its strip in it
  const LsopFastGeom& G = A.g;
  const int R = G.R, C = G.C, nS = G.nStrips, P = G.P;
  const int rbFloats = wave_rowbuf_floats(C);
  unsigned char* ring = waveSmem + size_t(warp) * (2 * kWaveChunkBytes);
  // rows 0 and 1 of this lane's tile (shared-memory address)
  const uint32_t rowbuf = smem_u32(waveSmem + size_t(kWaveWarps) * (2 * kWaveChunkBytes)) + uint32_t(warp * TPW + half) * uint32_t(2 * rbFloats) * 4u;
  uint64_t* bars = reinterpret_cast<uint64_t*>(waveSmem + size_t(kWaveWarps) * (2 * kWaveChunkBytes) +
                                               size_t(kWaveWarps * TPW) * (2 * rbFloats) * sizeof(float)) + 2 * warp;
  const uint32_t bar0 = smem_u32(bars);
  // this lane's residual bytes in ring stage 0 (lane 0: the start of the warp's ring)
  const uint32_t ringLane = smem_u32(ring) + uint32_t(half) * kHalfStage + uint32_t(ks * W);
  const bool isFirst = ks == 0, isLast = ks == nS - 1;
  if (lane == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;");
  }
  __syncwarp();
  // persistent warps: every warp fetches its next tile (pair of tiles) when it is through with one (no wave quantisation
  // of a static grid); gchunk counts the chunks this warp has fetched so far -- ring stage and mbarrier parity follow
  // from it across tiles
  uint32_t gchunk = 0;
  for (;;) {
  int li = 0;
  if (lane == 0) li = listBegin + atomicAdd(tileCounter, TPW);
  li = __shfl_sync(0xffffffffu, li, 0);
  if (li >= listEnd || li >= *a.listCount) break;
  // a tile that failed in kernel H, goes to the general path or was deferred by kernel T is skipped; so is the second
  // half of a pair at the end of the list.  A half without a tile stays idle while the other one works.
  li += half;
  int tIdx = 0, nExc = 0;
  bool live = false;
  if (!PAIR || (li < listEnd && li < *a.listCount)) {
    tIdx = a.list[li];
    if (a.status[tIdx] == G4_OK && *reinterpret_cast<const uint32_t*>(A.meta + size_t(tIdx) * kLsopMetaBytes) != 0u) {  // else general path
      nExc = int(A.exc[size_t(tIdx) * kExcWords]);
      live = nExc <= kExcCap;  // else deferred by kernel T
    }
  }
  const uint32_t liveMask = __ballot_sync(0xffffffffu, live);
  if (liveMask == 0u) continue;
  const bool anyExc = PAIR ? __any_sync(0xffffffffu, live && nExc > 0) : nExc > 0;  // (uniform)
  const bool active = live && ks < nS;
  const TileView t = tile_view(a.band, a.grid, tIdx);
  const uint32_t chunkBytes = uint32_t(CR * P);
  const int nChunks = G.nChunks;
  // image rows CR chunk .. CR chunk + CR - 1 into the next ring stage: lane 0 issues one copy per live tile (a skipped
  // tile may have no image) and one expect_tx for all of them.  Called by the whole warp; the second tile and the live
  // mask are fetched here rather than kept in registers across the steps.
  auto issue = [&](int chunk) {
    const uint32_t g = gchunk + uint32_t(chunk);
    const uint32_t bar = bar0 + 8u * (g & 1u), dst = ringLane + uint32_t(kWaveChunkBytes) * (g & 1u);  // (lane 0)
    const size_t off = size_t(chunk) * chunkBytes + kResidGuard;
    if constexpr (PAIR) {
      const int t1 = __shfl_sync(0xffffffffu, tIdx, 16);
      const uint32_t lm = __ballot_sync(0xffffffffu, live);
      if (lane == 0) {
        const bool l0 = (lm & 1u) != 0u, l1 = (lm >> 16) != 0u;
        mbar_expect_tx(bar, chunkBytes * uint32_t(int(l0) + int(l1)));
        if (l0)
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                       "l"(A.resid + size_t(tIdx) * size_t(G.tilePitch) + off), "r"(chunkBytes), "r"(bar)
                       : "memory");
        if (l1)
          asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst + kHalfStage),
                       "l"(A.resid + size_t(t1) * size_t(G.tilePitch) + off), "r"(chunkBytes), "r"(bar)
                       : "memory");
      }
    } else if (lane == 0) {
      mbar_expect_tx(bar, chunkBytes);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                   "l"(A.resid + size_t(tIdx) * size_t(G.tilePitch) + off), "r"(chunkBytes), "r"(bar)
                   : "memory");
    }
  };
  issue(0);

  float u[12];
#pragma unroll
  for (int i = 0; i < 12; i++) u[i] = active ? A.coef[size_t(tIdx) * 12 + i] : 0.f;
  // rows 0 and 1 as floats (int -> float exactly as the reference converts them)
  if (live)
    for (int c = ks; c < rbFloats; c += HL) {
      const float x = c < C ? float(t.row(0)[c]) : 0.f, y = c < C ? float(t.row(1)[c]) : 0.f;
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(rowbuf + 4u * uint32_t(c)), "f"(x) : "memory");
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(rowbuf + 4u * uint32_t(rbFloats + c)), "f"(y) : "memory");
    }
  // side records: the first lane needs {v[r][0], v[r][1]} of each, the last lane {D2[r], D1[r]} (nStrips >= 2)
  const int2* side = reinterpret_cast<const int2*>(A.side + size_t(tIdx) * R) + (isLast ? 1 : 0);
  const bool needSide = active && (isFirst || isLast);
  // rr = (row this lane works on in the coming step) - 2; lanes that hold no strip never become valid
  uint32_t rr = active ? uint32_t(-ks) : 0x40000000u;
  const uint32_t nRowsIn = uint32_t(R - 2);
  int2 sideCur = make_int2(0, 0), sideNext = make_int2(0, 0);
  if (needSide && rr < nRowsIn) sideNext = side[2 * (2 + rr)];  // (first lane; the last lane fetches when its rows begin)
  const int2* sideAt = side + 2 * (3 - ks);                      // record of the row after the coming step's (dereferenced for valid rows)
  char* rowp = reinterpret_cast<char*>(t.base + int64_t(2 - ks) * t.pitch + ks * W);  // dereferenced only for valid rows
  const int64_t rowStep = int64_t(t.pitch) * 4;
  uint32_t ringAt = ringLane;                             // this lane's residual bytes of the coming step
  const uint32_t rb0 = rowbuf + uint32_t(ks * W) * 4u, rb1 = rb0 + uint32_t(rbFloats) * 4u;
  const int wInterior = C - 4;
  uint32_t badBits = 0;  // nonzero: some cell left the range of the fast arithmetic
  float a0[W + 4], a1[W + 4], a2[W + 4];  // three rows of the strip, columns 2 + kW - 2 .. 2 + kW + W + 1, rotating roles
#pragma unroll
  for (int i = 0; i < W + 4; i++) { a0[i] = 0.f; a1[i] = 0.f; a2[i] = 0.f; }
  int32_t pa = 0, pb = 0;        // own outputs of cells W - 2, W - 1 of the previous step (the right neighbour's left values)
  __syncwarp();

  // one step: row r of the strip into cur[]; am1 / am2 hold rows r - 1 / r - 2
  auto step = [&](float (&am2)[W + 4], float (&am1)[W + 4], float (&cur)[W + 4], const int s) {
    if ((s & (CR - 1)) == 0) {  // (uniform) next chunk of the residual image
      const int chunk = s / CR;
      if (chunk < nChunks) {
        if (chunk + 1 < nChunks) issue(chunk + 1);
        const uint32_t g = gchunk + uint32_t(chunk);
        mbar_wait(bar0 + 8u * (g & 1u), (g >> 1) & 1u);
      }
      ringAt = ringLane + uint32_t(kWaveChunkBytes) * ((gchunk + uint32_t(chunk)) & 1u);
    }
    const bool valid = rr < nRowsIn;
    const bool first = rr == 0u;
    if (s < nS) {  // (uniform) the steps in which some lane begins
     if (first) {  // (one lane per step) rows 0 and 1 from the row buffer
#pragma unroll
      for (int i = 0; i < W + 4; i += 4) {
        float4 x, y;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w) : "r"(rb0 + 4u * i));
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(y.x), "=f"(y.y), "=f"(y.z), "=f"(y.w) : "r"(rb1 + 4u * i));
        am2[i] = x.x; am2[i + 1] = x.y; am2[i + 2] = x.z; am2[i + 3] = x.w;
        am1[i] = y.x; am1[i + 1] = y.y; am1[i + 2] = y.z; am1[i + 3] = y.w;
      }
     }
    }
    // side record of this row (first lane: columns 0,1; last lane: D2, D1), the next row's fetched now
    sideCur = sideNext;
    if (needSide && rr + 1u < nRowsIn) sideNext = *sideAt;
    sideAt += 2;
    // residual bytes of the strip
    uint32_t rw[NW];
    {
      const uint32_t at = ringAt;
      ringAt += uint32_t(P);
      if constexpr (NW == 1) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(rw[0]) : "r"(at));
      else if constexpr (NW == 2) asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(rw[0]), "=r"(rw[1]) : "r"(at));
      else asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(rw[0]), "=r"(rw[1]), "=r"(rw[2]), "=r"(rw[3]) : "r"(at));
    }
    // left values: cells W-2, W-1 of row r in the strip to the left (finished one step ago: its am1), or columns 0,1
    float l2 = __shfl_up_sync(0xffffffffu, am1[W], 1, HL), l1 = __shfl_up_sync(0xffffffffu, am1[W + 1], 1, HL);
    int32_t li2 = __shfl_up_sync(0xffffffffu, pa, 1, HL), li1 = __shfl_up_sync(0xffffffffu, pb, 1, HL);
    if (isFirst) { li2 = sideCur.x; li1 = sideCur.y; l2 = float(li2); l1 = float(li1); }
    cur[0] = l2;
    cur[1] = l1;
    // exceptions: a zero byte in a tile that has an exception list -> the general form of the step (for the whole warp)
    bool general = false;
    if (anyExc) {
      bool z = false;
#pragma unroll
      for (int i = 0; i < NW; i++) z = z || ((rw[i] - 0x01010101u) & ~rw[i] & 0x80808080u) != 0u;
      general = __any_sync(0xffffffffu, z && valid);
    }
    int32_t oi[W];
    auto store_lo = [&](const int32_t (&o)[W]) {  // columns k W .. k W + 7 of the raster row: {left2, left1, cells 0 .. 5}
      if constexpr (W >= 8) {
        if (WIDE) {
          asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(rowp), "r"(li2), "r"(li1), "r"(o[0]), "r"(o[1]), "r"(o[2]),
                       "r"(o[3]), "r"(o[4]), "r"(o[5])
                       : "memory");
        } else {
          *reinterpret_cast<int4*>(rowp) = make_int4(li2, li1, o[0], o[1]);
          *reinterpret_cast<int4*>(rowp + 16) = make_int4(o[2], o[3], o[4], o[5]);
        }
      }
    };
    uint32_t accLo = 0, accHi = 0;  // exponent bits of t1 that differ from those of [2^22, 2^23): nonzero <=> p outside [-2^21, 2^21) or NaN
    auto cells = [&](auto genTag) {
      constexpr bool GEN = decltype(genTag)::value;
#pragma unroll
      for (int j = 0; j < W; j++) {
        constexpr int dummy = 0;
        (void)dummy;
        const int c = j + 2;
        if (j == 2) {  // cells 0,1 of row r - 1 in the strip to the right were computed a moment ago (its cur[2], cur[3])
          const float s0 = __shfl_down_sync(0xffffffffu, cur[2], 1, HL), s1 = __shfl_down_sync(0xffffffffu, cur[3], 1, HL);
          if (!first) {  // (in its first step the lane has row 1 right of the strip from the row buffer)
            am1[W + 2] = s0;
            am1[W + 3] = s1;
          }
        }
        // LsDecoder12.java:424-438 -- evaluated left to right in float32, no fused multiply-add
        float p = u[0] * cur[c - 1];
        p = p + u[1] * am1[c - 1];
        p = p + u[2] * am1[c];
        p = p + u[3] * am1[c + 1];
        p = p + u[4] * am1[c + 2];
        p = p + u[5] * cur[c - 2];
        p = p + u[6] * am1[c - 2];
        p = p + u[7] * am2[c - 2];
        p = p + u[8] * am2[c - 1];
        p = p + u[9] * am2[c];
        p = p + u[10] * am2[c + 1];
        p = p + u[11] * am2[c + 2];
        const float t1 = __fadd_rd(p, kMagicHalf);
        if (j < E) accLo |= __float_as_uint(t1) ^ 0x4A800000u;
        else accHi |= __float_as_uint(t1) ^ 0x4A800000u;
        const float t2 = __fadd_rd(t1, kMagicHalfUp);  // 1.5*2^23 + StrictMath.round(p)
        const uint32_t word = rw[j >> 2];
        const float xj = __uint_as_float(__byte_perm(word, 0x4B400000u, 0x7640 + (j & 3)));  // 1.5*2^23 + residual + 128
        float fv = t2 + (xj - (2.f * kMagicInt + 128.f));  // exact: float(round(p) + residual)
        int32_t iv;
        if constexpr (GEN) {
          const uint32_t byte = (word >> (8 * (j & 3))) & 0xffu;
          int32_t ex = int32_t(byte) - 128;
          if (byte == 0u && valid) ex = wave_exception(A.exc + size_t(tIdx) * kExcWords, int(rr) * wInterior + ks * W + j);
          iv = int32_t(uint32_t(__float_as_int(t2)) - 0x4B400000u + uint32_t(ex));
          fv = float(iv);
        } else iv = int32_t(uint32_t(__float_as_int(t2)) + __float_as_uint(xj) - 0x96800080u);  // round(p) + byte - 128
        if (j == E || j == E + 1) {  // the last strip: Triangle predictor folded into D2 / D1 by kernel H (LsDecoder12.java:459-468)
          const int32_t prev = j == 0 ? li1 : oi[j > 0 ? j - 1 : 0];
          const int32_t sv = int32_t(uint32_t(prev) + uint32_t(j == E ? sideCur.x : sideCur.y));
          if (isLast) { iv = sv; fv = float(sv); }
        }
        oi[j] = iv;
        cur[c] = fv;
        if (kEarlyLo && j == 5 && valid) store_lo(oi);  // (frees oi[0 .. 5] for the second half of the strip)
      }
    };
    if (general) cells(std::true_type{});
    else cells(std::false_type{});
    if (valid) badBits |= (accLo | (isLast ? 0u : accHi)) & 0xFF800000u;
    // raster: columns k W .. k W + W - 1 of row r = {left2, left1, cells 0 .. W - 3}
    if (valid) {
      if constexpr (W == 4) *reinterpret_cast<int4*>(rowp) = make_int4(li2, li1, oi[0], oi[1]);
      else {
        if constexpr (!kEarlyLo) store_lo(oi);
        if constexpr (W == 16) {
          if (WIDE) {
            asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(rowp + 32), "r"(oi[6]), "r"(oi[7]), "r"(oi[8]), "r"(oi[9]),
                         "r"(oi[10]), "r"(oi[11]), "r"(oi[12]), "r"(oi[13])
                         : "memory");
          } else {
            *reinterpret_cast<int4*>(rowp + 32) = make_int4(oi[6], oi[7], oi[8], oi[9]);
            *reinterpret_cast<int4*>(rowp + 48) = make_int4(oi[10], oi[11], oi[12], oi[13]);
          }
        }
      }
    }
    pa = oi[W - 2];
    pb = oi[W - 1];
    rr++;
    rowp += rowStep;
    __syncwarp();
  };

  const int nSteps = G.nSteps;
#pragma unroll 1
  for (int s = 0; s < nSteps; s += 3) {
    step(a0, a1, a2, s);
    step(a1, a2, a0, s + 1);
    step(a2, a0, a1, s + 2);
  }
  // outside the fast arithmetic's range: the general kernels redo the tile
  const uint32_t bad = __ballot_sync(0xffffffffu, badBits != 0u);
  if (isFirst && (PAIR ? (bad >> (16 * half)) & 0xffffu : bad) != 0u) A.defer[atomicAdd(A.deferCount, 1)] = tIdx;
  gchunk += uint32_t(nChunks);
  }
}

size_t head_smem_bytes(const LsopFastGeom& g) {
  const size_t nInit = size_t(4 * g.R + 2 * g.C - 9);
  return size_t(kWarps) * (((sizeof(CanonWarpShared) + 15) & ~size_t(15)) + ((nInit * 4 + 15) & ~size_t(15))) + 16;
}
uint32_t text_stage_words(const LsopFastGeom& g) {
  // 5 bits per sample of the tile plus the headers, at least 2 KB (a packing that does not fit goes to the general kernels)
  uint32_t w = uint32_t((uint64_t(g.R) * uint64_t(g.C) * 5 / 8 + 3) / 4) + 128u;
  if (w < 512u) w = 512u;
  return (w + 255u) & ~255u;
}
size_t text_smem_bytes(const LsopFastGeom& g) { return text_fast_bytes(text_stage_words(g)) + size_t(g.tileBytes); }
bool text_small(const LsopFastGeom& g) { return uint32_t(g.R) * uint32_t(g.C) <= kTextSmallTile; }
size_t wave_smem_bytes(const LsopFastGeom& g) {
  const size_t rbFloats = size_t((g.C + 4 + 3) & ~3);
  return size_t(kWaveWarps) * (2 * kWaveChunkBytes) + size_t(kWaveWarps * g.tilesPerWarp) * (2 * rbFloats) * sizeof(float) +
         size_t(kWaveWarps) * 16;
}

template <int W, bool WIDE, bool PAIR>
cudaError_t launch_wave_kernel(const LsopFastArgs& A, int nCtas, int nTilesUpper, int* tileCounter, cudaStream_t s) {
  const size_t smem = wave_smem_bytes(A.g);
  cudaError_t e = cudaFuncSetAttribute(lsop3_wave_kernel<W, WIDE, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  if (e != cudaSuccess) return e;
  lsop3_wave_kernel<W, WIDE, PAIR><<<nCtas, 32 * kWaveWarps, smem, s>>>(A, tileCounter, 0, nTilesUpper);
  return cudaGetLastError();
}
template <int W>
cudaError_t launch_wave(const LsopFastArgs& A, int nCtas, int nTilesUpper, int* tileCounter, cudaStream_t s) {
  if (A.g.tilesPerWarp == 2)
    return A.g.wide ? launch_wave_kernel<W, true, true>(A, nCtas, nTilesUpper, tileCounter, s)
                    : launch_wave_kernel<W, false, true>(A, nCtas, nTilesUpper, tileCounter, s);
  return A.g.wide ? launch_wave_kernel<W, true, false>(A, nCtas, nTilesUpper, tileCounter, s)
                  : launch_wave_kernel<W, false, false>(A, nCtas, nTilesUpper, tileCounter, s);
}

}  // namespace

bool lsop_fast_geometry(const g4_band_desc& band, const void* grid, LsopFastGeom* out) {
  LsopFastGeom g{};
  g.R = band.tile_rows;
  g.C = band.tile_cols;
  if (g.R < 6 || g.C < 16 || (g.C & 3) != 0 || (band.grid_pitch & 3) != 0 || (reinterpret_cast<uintptr_t>(grid) & 15) != 0) return false;
  // strip width: C has to be a multiple of it (the last strip then ends with the row's last two columns).  The narrowest
  // that covers the columns with 16 lanes, two tiles per warp: fewer ramp steps per tile, more cells per step to share
  // the fixed cost of a step, and 30 of 32 lanes busy at 240 columns instead of 30 (W 8, 207 steps for 178 rows) or
  // 15 (W 16 single).  Otherwise the narrowest that covers them with 32 lanes, one tile per warp.
  g.tilesPerWarp = 1;
  for (int w = 4; w <= 16; w *= 2)
    if (g.C % w == 0 && (g.C - 2 + w - 1) / w <= 16) {
      g.W = w;
      g.tilesPerWarp = 2;
      break;
    }
  if (g.tilesPerWarp == 1) {
    if (g.C <= 128) g.W = 4;
    else if (g.C <= 256 && (g.C & 7) == 0) g.W = 8;
    else if (g.C <= 512 && (g.C & 15) == 0) g.W = 16;
    else return false;
  }
  g.logW = g.W == 4 ? 2 : g.W == 8 ? 3 : 4;
  g.nStrips = (g.C - 2 + g.W - 1) / g.W;
  g.P = g.nStrips * g.W;
  g.nSteps = g.R - 2 + g.nStrips - 1;
  g.chunkRows = 128 / g.W;
  g.nChunks = (g.nSteps + g.chunkRows - 1) / g.chunkRows;
  g.tileBytes = g.nChunks * g.chunkRows * g.P;  // a multiple of 128
  g.tilePitch = g.tileBytes;
  g.wide = ((band.grid_pitch & 7) == 0 && (reinterpret_cast<uintptr_t>(grid) & 31) == 0) ? 1 : 0;
  if (text_smem_bytes(g) > 224u * 1024u || head_smem_bytes(g) > 224u * 1024u || wave_smem_bytes(g) > 224u * 1024u) return false;
  *out = g;
  return true;
}
size_t lsop_fast_side_bytes(const LsopFastGeom& g, int nTiles) { return size_t(nTiles) * size_t(g.R) * sizeof(int4); }
size_t lsop_fast_exc_bytes(int nTiles) { return size_t(nTiles) * kExcWords * sizeof(uint32_t); }
size_t lsop_fast_stage_bytes(int smCount) { return size_t(smCount) * 4 * kFastMaxSub * kSpillWords * sizeof(uint32_t); }  // text kernel: <= 4 CTAs per SM
size_t lsop_fast_resid_bytes(const LsopFastGeom& g, int nTiles) { return size_t(kResidGuard) + size_t(nTiles) * size_t(g.tilePitch) + 4096; }

// Kernels H, T and W over the list positions [0, nTilesUpper).  Tiles the fast path cannot take are appended to
// A.defer / A.deferCount for the general kernels, which the caller launches AFTER this returns.
// The kernels take that range as [listBegin, listEnd) arguments: compiled without them, kernel T keeps its shared-memory
// addresses in vector instead of uniform registers, and the config-3 decode measured up to 0.2 % slower (B200, 1000 W).
cudaError_t launch_lsop_decode_fast(const LsopFastArgs& A, int nTilesUpper, int smCount, int* textCounter, cudaStream_t s, int* launches) {
  const LsopFastGeom& g = A.g;
  // dynamic shared memory opt-in: per device and per geometry, so simply set before every launch set (host-side only)
  {
    cudaError_t e = cudaFuncSetAttribute(lsop2_head_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(head_smem_bytes(g)));
    if (e == cudaSuccess)
      e = text_small(g) ? cudaFuncSetAttribute(lsop2_text_kernel<kTextThreadsSmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(text_smem_bytes(g)))
                        : cudaFuncSetAttribute(lsop2_text_kernel<kTextThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(text_smem_bytes(g)));
    if (e != cudaSuccess) return e;
  }
  const uint32_t stageWords = text_stage_words(g);
  const int nCtasWarp = (nTilesUpper + kWarps - 1) / kWarps;
  lsop2_head_kernel<<<nCtasWarp, kThreads, head_smem_bytes(g), s>>>(A, stageWords * 4u, 0, nTilesUpper);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  LsopFastArgs T = A;
  T.a.counter = textCounter;
  const size_t textSmem = text_smem_bytes(g);
  int perSm = int((227u * 1024u) / (textSmem + 1024));
  const int perSmCap = text_small(g) ? 4 : 2;  // 64 registers per thread: 1,024 threads per SM
  if (perSm < 1) perSm = 1;
  if (perSm > perSmCap) perSm = perSmCap;
  int ctas = smCount * perSm;
  if (ctas > nTilesUpper) ctas = nTilesUpper;
  if (text_small(g)) lsop2_text_kernel<kTextThreadsSmall><<<ctas, kTextThreadsSmall, textSmem, s>>>(T, stageWords, 0, nTilesUpper);
  else lsop2_text_kernel<kTextThreads><<<ctas, kTextThreads, textSmem, s>>>(T, stageWords, 0, nTilesUpper);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  const int nWarpsWave = (nTilesUpper + g.tilesPerWarp - 1) / g.tilesPerWarp;
  int nCtasWave = (nWarpsWave + kWaveWarps - 1) / kWaveWarps;
  if (nCtasWave > smCount * G4_WAVE_CTAS) nCtasWave = smCount * G4_WAVE_CTAS;  // persistent: one resident set of CTAs
  int* waveCounter = textCounter + 1;
  e = g.W == 4 ? launch_wave<4>(A, nCtasWave, nTilesUpper, waveCounter, s) : g.W == 8 ? launch_wave<8>(A, nCtasWave, nTilesUpper, waveCounter, s)
                                                                                          : launch_wave<16>(A, nCtasWave, nTilesUpper, waveCounter, s);
  if (e != cudaSuccess) return e;
  if (launches) *launches += 3;
  return cudaSuccess;
}

}  // namespace g4
