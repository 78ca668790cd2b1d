// g4_records.cu -- GVRS tile records on the device: framing, CRC-32C, and the inverse (payload location + checksum check).
//
// Reference (under /root/reference/core/src/main/java/org/gridfour/):
//   gvrs/RecordManager.java:70-78      record = [size:int32 LE][type:uint8][0,0,0] content, zero padding, [crc32c:int32 LE];
//                                      RECORD_HEADER_SIZE 8, RECORD_OVERHEAD_SIZE 12
//   gvrs/RecordManager.java:137-139    sizes are rounded up to a multiple of 8 (multipleOf8)
//   gvrs/RecordManager.java:161-204    fileSpaceInitRecord / fileSpaceFinishRecord: header, zero fill, CRC over the first
//                                      size-4 bytes of the record when checksums are enabled (the field stays 0 otherwise)
//   gvrs/RecordManager.java:386-490    writeTile: content = [tileIndex:int32] then per element [len:int32][bytes]
//   gvrs/RecordManager.java:492-516    readTile: len == standard size -> raw element, else a codec packing
//   gvrs/RecordType.java:43-51         Tile = 2
//   util/GridfourCRC32C.java:156-163   CRC-32C (Castagnoli, reflected, init/final xor 0xffffffff), byte-wise table form
//
// record_pack_kernel / record_unpack_kernel frame and read the records of rasters with ONE element per tile
// (content = [tileIndex][len][payload], payload 8-byte aligned on both sides).  record_pack_multi_kernel /
// record_unpack_multi_kernel do the same for any number of elements ([tileIndex] then [len_e][payload_e] per element, every
// payload after the first at any byte offset); both reuse record_layout_kernel and crc32c_kernel.  g4_crc32c is general
// and serves every record type.
#include "g4_kernels.h"
#include "g4_device.cuh"

namespace g4 {

namespace {

constexpr int kCrcThreads = 128;
constexpr uint32_t kCrc32cPoly = 0x82F63B78u;  // reflected Castagnoli polynomial; table entry 1 is 0xf26b8303 as in the reference

// Slice-by-8 tables in shared memory: T[0] is the reference's CRC_TABLE, T[k][i] = (T[k-1][i] >> 8) ^ T[0][T[k-1][i] & 255].
__device__ inline void crc_build_tables(uint32_t (*T)[256]) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint32_t c = uint32_t(i);
#pragma unroll
    for (int k = 0; k < 8; k++) c = (c >> 1) ^ ((c & 1u) ? kCrc32cPoly : 0u);
    T[0][i] = c;
  }
  __syncthreads();
  for (int k = 1; k < 8; k++) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
      const uint32_t p = T[k - 1][i];
      T[k][i] = (p >> 8) ^ T[0][p & 0xffu];
    }
    __syncthreads();
  }
}

__device__ inline uint32_t crc_range(const uint32_t (*T)[256], const uint8_t* p, uint32_t n) {
  uint32_t c = 0xffffffffu;
  while (n && (reinterpret_cast<uintptr_t>(p) & 7)) {
    c = T[0][(c ^ *p++) & 0xffu] ^ (c >> 8);
    n--;
  }
  const uint2* q = reinterpret_cast<const uint2*>(p);
  for (; n >= 8; n -= 8) {
    const uint2 v = *q++;
    const uint32_t a = v.x ^ c, b = v.y;
    c = T[7][a & 0xffu] ^ T[6][(a >> 8) & 0xffu] ^ T[5][(a >> 16) & 0xffu] ^ T[4][a >> 24] ^ T[3][b & 0xffu] ^ T[2][(b >> 8) & 0xffu] ^
        T[1][(b >> 16) & 0xffu] ^ T[0][b >> 24];
  }
  p = reinterpret_cast<const uint8_t*>(q);
  while (n--) c = T[0][(c ^ *p++) & 0xffu] ^ (c >> 8);
  return c ^ 0xffffffffu;
}

}  // namespace

// GF(2) arithmetic for joining the CRCs of adjacent pieces (the construction of zlib's crc32_combine, with the
// Castagnoli polynomial): crc(A||B) = crc(A) * x^(8|B|) mod P  xor  crc(B).
__device__ inline uint32_t crc_multmodp(uint32_t a, uint32_t b) {
  uint32_t m = 1u << 31, p = 0;
  for (;;) {
    if (a & m) {
      p ^= b;
      if ((a & (m - 1u)) == 0) break;
    }
    m >>= 1;
    b = (b & 1u) ? (b >> 1) ^ kCrc32cPoly : b >> 1;
  }
  return p;
}
// x^(n * 2^k) mod P from the table of x^(2^i) mod P
__device__ inline uint32_t crc_x2nmodp(const uint32_t* x2n, uint64_t n, uint32_t k) {
  uint32_t p = 1u << 31;  // x^0
  while (n) {
    if (n & 1u) p = crc_multmodp(x2n[k & 31u], p);
    n >>= 1;
    k++;
  }
  return p;
}

// One WARP per byte range (ranges are whole records: a few KB to a few hundred KB each, thousands per launch): every
// lane takes a contiguous piece (a multiple of 8 bytes, so that the slice-by-8 loop stays aligned), the 32 piece CRCs
// are joined by a shuffle tree in which level d multiplies the left CRC by x^(8 * piece * 2^d).
// storeAtEnd: also write the value, little-endian, into the four bytes that follow the range (the record's checksum field).
__global__ void __launch_bounds__(kCrcThreads) crc32c_kernel(const uint8_t* data, const uint64_t* offsets, const uint32_t* sizes, int n,
                                                             uint32_t* out, int storeAtEnd) {
  __shared__ uint32_t T[8][256];
  __shared__ uint32_t x2n[32];
  crc_build_tables(T);
  if (threadIdx.x == 0) {
    uint32_t p = 1u << 30;  // x^1
    x2n[0] = p;
    for (int i = 1; i < 32; i++) x2n[i] = p = crc_multmodp(p, p);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * kCrcThreads + threadIdx.x) >> 5;
  if (i >= n) return;
  const uint8_t* p = data + offsets[i];
  const uint32_t len = sizes[i];
  // piece size: a multiple of 8, at least 64 bytes; short ranges leave the upper lanes with nothing
  uint32_t piece = ((len + 31u) / 32u + 7u) & ~7u;
  if (piece < 64u) piece = 64u;
  const uint64_t begin = uint64_t(lane) * piece;
  const uint32_t mine = begin >= len ? 0u : (len - begin < piece ? uint32_t(len - begin) : piece);
  uint32_t c = crc_range(T, p + begin, mine);  // CRC of an empty piece is 0, the identity of the join
  uint32_t myLen = mine;
  // join: after level d, lanes that are multiples of 2^(d+1) hold the CRC of 2^(d+1) pieces
#pragma unroll
  for (int d = 0; d < 5; d++) {
    const uint32_t rc = __shfl_down_sync(0xffffffffu, c, 1u << d);
    const uint32_t rl = __shfl_down_sync(0xffffffffu, myLen, 1u << d);
    if ((lane & ((2 << d) - 1)) == 0 && rl) {
      c = crc_multmodp(crc_x2nmodp(x2n, rl, 3), c) ^ rc;
      myLen += rl;
    }
  }
  if (lane == 0) {
    if (out) out[i] = c;
    if (storeAtEnd) {
      uint8_t* e = const_cast<uint8_t*>(p) + len;
      e[0] = uint8_t(c); e[1] = uint8_t(c >> 8); e[2] = uint8_t(c >> 16); e[3] = uint8_t(c >> 24);
    }
  }
}

// LSOP12 value checksum (LsHeader.computeChecksum :391-406, checked in LsDecoder12.decode :153-158): CRC-32C of the tile's
// nRows x nColumns values as little-endian int32, row-major.  One WARP per tile of the list whose packing carries the
// checksum; every lane takes a contiguous run of values (an even number: the slice-by-8 step eats two), the 32 pieces are
// joined like in crc32c_kernel.  The tile is a strided window of the raster, so the values are read cell by cell.
__global__ void __launch_bounds__(kCrcThreads) lsop_value_checksum_kernel(DecodeArgs a) {
  __shared__ uint32_t T[8][256];
  __shared__ uint32_t x2n[32];
  const int lane = threadIdx.x & 31;
  const int li = (blockIdx.x * kCrcThreads + threadIdx.x) >> 5;
  // (uniform per warp) does this warp's tile carry a checksum at all?  Most files do not: leave before building the tables.
  bool need = false;
  int tIdx = 0;
  if (li < *a.listCount) {
    tIdx = a.list[li];
    need = a.lsopCks[2 * tIdx] != 0u && a.status[tIdx] == G4_OK;
  }
  if (!__syncthreads_or(need ? 1 : 0)) return;
  crc_build_tables(T);
  if (threadIdx.x == 0) {
    uint32_t p = 1u << 30;  // x^1
    x2n[0] = p;
    for (int i = 1; i < 32; i++) x2n[i] = p = crc_multmodp(p, p);
  }
  __syncthreads();
  if (!need) return;
  const TileView t = tile_view(a.band, a.grid, tIdx);
  const uint32_t n = uint32_t(t.R) * uint32_t(t.C);
  uint32_t piece = ((n + 31u) / 32u + 1u) & ~1u;
  if (piece < 16u) piece = 16u;
  const uint32_t begin = uint32_t(lane) * piece;
  const uint32_t mine = begin >= n ? 0u : (n - begin < piece ? n - begin : piece);
  uint32_t c = 0xffffffffu;
  {
    int r = int(begin / uint32_t(t.C)), col = int(begin - uint32_t(r) * uint32_t(t.C));
    const int32_t* row = t.row(r < t.R ? r : 0);
    auto next = [&]() {
      const uint32_t v = uint32_t(row[col]);
      if (++col == t.C) { col = 0; row += t.pitch; }
      return v;
    };
    uint32_t k = 0;
    for (; k + 2 <= mine; k += 2) {
      const uint32_t a0 = next() ^ c, b0 = next();
      c = T[7][a0 & 0xffu] ^ T[6][(a0 >> 8) & 0xffu] ^ T[5][(a0 >> 16) & 0xffu] ^ T[4][a0 >> 24] ^ T[3][b0 & 0xffu] ^ T[2][(b0 >> 8) & 0xffu] ^
          T[1][(b0 >> 16) & 0xffu] ^ T[0][b0 >> 24];
    }
    if (k < mine) {
      uint32_t v = next();
      for (int i = 0; i < 4; i++, v >>= 8) c = T[0][(c ^ v) & 0xffu] ^ (c >> 8);
    }
  }
  c = mine ? c ^ 0xffffffffu : 0u;  // CRC of an empty piece is 0, the identity of the join
  uint32_t myLen = 4u * mine;
#pragma unroll
  for (int d = 0; d < 5; d++) {
    const uint32_t rc = __shfl_down_sync(0xffffffffu, c, 1u << d);
    const uint32_t rl = __shfl_down_sync(0xffffffffu, myLen, 1u << d);
    if ((lane & ((2 << d) - 1)) == 0 && rl) {
      c = crc_multmodp(crc_x2nmodp(x2n, rl, 3), c) ^ rc;
      myLen += rl;
    }
  }
  if (lane == 0 && c != a.lsopCks[2 * tIdx + 1]) a.status[tIdx] = G4_CHECKSUM_MISMATCH;
}

cudaError_t launch_lsop_value_checksum(const DecodeArgs& a, int nTilesUpper, cudaStream_t s) {
  const int warpsPerCta = kCrcThreads / 32;
  lsop_value_checksum_kernel<<<(nTilesUpper + warpsPerCta - 1) / warpsPerCta, kCrcThreads, 0, s>>>(a);
  return cudaGetLastError();
}

// Record sizes and positions of a batch of single-element tile records: size = multipleOf8(12 + 4 + 4 + len), exclusive
// scan from basePos.  contentPos[t] = record position + 8 (what the tile directory stores, RecordManager.java:218-219);
// crcOff/crcLen describe the checksummed part of every record relative to `records`.  One CTA.
__global__ void __launch_bounds__(kThreads) record_layout_kernel(const uint32_t* lens, int n, uint64_t basePos, uint64_t* contentPos,
                                                                 uint64_t* crcOff, uint32_t* crcLen, uint64_t* total) {
  __shared__ unsigned long long sm[kWarps];
  __shared__ unsigned long long carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int t0 = 0; t0 < n; t0 += kThreads) {
    const int t = t0 + threadIdx.x;
    const unsigned long long x = t < n ? ((unsigned long long)(lens[t]) + 12ull + 8ull + 7ull) & ~7ull : 0ull;
    unsigned long long inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const unsigned long long y = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += y;
    }
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    unsigned long long base = carry;
    for (int w = 0; w < warp; w++) base += sm[w];
    if (t < n) {
      const unsigned long long rec = base + inc - x;
      contentPos[t] = basePos + rec + 8ull;
      crcOff[t] = rec;
      crcLen[t] = uint32_t(x - 4ull);
    }
    __syncthreads();
    if (threadIdx.x == kThreads - 1) carry = base + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

// One CTA per tile: header, tile index, payload length, payload (both sides 8-byte aligned), zero padding and a zero
// checksum field (crc32c_kernel fills it in when checksums are enabled).
__global__ void __launch_bounds__(kThreads) record_pack_kernel(const uint8_t* arena, const uint64_t* offsets, const uint32_t* lens,
                                                               const int32_t* tileIndex, int firstTileIndex, int n, const uint64_t* crcOff,
                                                               const uint32_t* crcLen, uint8_t* records) {
  for (int t = blockIdx.x; t < n; t += gridDim.x) {
    uint8_t* rec = records + crcOff[t];
    const uint32_t size = crcLen[t] + 4u, len = lens[t];
    uint32_t* w = reinterpret_cast<uint32_t*>(rec);
    if (threadIdx.x == 0) {
      w[0] = size;
      w[1] = 2u;  // RecordType.Tile, three reserved zero bytes
      w[2] = uint32_t(tileIndex ? tileIndex[t] : firstTileIndex + t);
      w[3] = len;
    }
    const uint8_t* src = arena + offsets[t];
    uint8_t* dst = rec + 16;
    const uint32_t span = size - 16u;  // payload + padding + checksum field
    if ((reinterpret_cast<uintptr_t>(src) & 3) == 0) {
      const uint32_t* s4 = reinterpret_cast<const uint32_t*>(src);
      uint32_t* d4 = reinterpret_cast<uint32_t*>(dst);
      const uint32_t full = len >> 2;
      for (uint32_t i = threadIdx.x; i < (span >> 2); i += kThreads) {
        uint32_t v = 0;
        if (i < full) v = s4[i];
        else if (i == full && (len & 3)) {
          for (uint32_t b = 0; b < (len & 3); b++) v |= uint32_t(src[full * 4 + b]) << (8 * b);
        }
        d4[i] = v;
      }
    } else {
      for (uint32_t i = threadIdx.x; i < span; i += kThreads) dst[i] = i < len ? src[i] : uint8_t(0);
    }
  }
}

// One thread per tile: checks the record around contentPos[t] (RecordManager.readTile :492-516 trusts the file; a GPU
// reader must not) and returns where the element payload sits inside the image.
__global__ void __launch_bounds__(kThreads) record_unpack_kernel(const uint8_t* image, uint64_t imageLen, const uint64_t* contentPos, int n,
                                                                 uint64_t* payloadOff, uint32_t* lens, uint64_t* crcOff, uint32_t* crcLen,
                                                                 uint32_t* storedCrc, int32_t* status) {
  const int t = blockIdx.x * kThreads + threadIdx.x;
  if (t >= n) return;
  const uint64_t cp = contentPos[t];
  int st = G4_OK;
  uint64_t po = 0;
  uint32_t ln = 0, cl = 0, sc = 0;
  uint64_t co = 0;
  if (cp == 0) st = G4_DECLINED;  // tile not present in the file (directory entry 0, RecordManager.java:495-498)
  else if ((cp & 7) || cp < 8 || cp + 8 > imageLen) st = G4_ERR_FORMAT;
  else {
    const uint32_t* h = reinterpret_cast<const uint32_t*>(image + cp - 8);
    const uint32_t size = h[0];
    const uint32_t type = h[1] & 0xffu;
    ln = h[3];
    if (type != 2u || size < 24u || (size & 7u) || cp - 8 + size > imageLen || uint64_t(ln) + 20ull > size) st = G4_ERR_FORMAT;
    else {
      po = cp + 8;
      co = cp - 8;
      cl = size - 4u;
      sc = *reinterpret_cast<const uint32_t*>(image + cp - 8 + size - 4);
    }
  }
  payloadOff[t] = po;
  lens[t] = st == G4_OK ? ln : 0u;
  crcOff[t] = co;
  crcLen[t] = cl;
  storedCrc[t] = sc;
  status[t] = st;
}

__global__ void __launch_bounds__(kThreads) record_verify_kernel(const uint32_t* computed, const uint32_t* stored, int n, int32_t* status) {
  const int t = blockIdx.x * kThreads + threadIdx.x;
  if (t >= n) return;
  if (status[t] == G4_OK && computed[t] != stored[t]) status[t] = G4_ERR_FORMAT;
}

// ---- tile records of rasters with several elements per tile -----------------------------------------------------------
// content = [tileIndex] then, per element e, [len_e][len_e bytes]; size = multipleOf8(12 + 4 + sum_e(4 + len_e)).
// record_layout_kernel computes that size from chainLens[t] = sum_e(4 + len_e) - 4 (its own rounding adds the 20 bytes of
// header, tile index, first length field and checksum field).

// Four bytes from any address: the two aligned words around it joined by a funnel shift.  The second word is read only
// when p is misaligned, and then it holds p[3], so it never leaves the granule of a byte the caller owns.
__device__ inline uint32_t load_u32_funnel(const uint8_t* p) {
  const uint32_t sh = uint32_t(reinterpret_cast<uintptr_t>(p) & 3u);
  const uint32_t* a = reinterpret_cast<const uint32_t*>(p - sh);
  const uint32_t lo = a[0];
  return sh ? __funnelshift_r(lo, a[1], 8u * sh) : lo;
}

// One thread per tile.
__global__ void __launch_bounds__(kThreads) record_chain_lens_kernel(const RecordElement* elems, int nElements, int n,
                                                                     uint32_t* chainLens) {
  const int t = blockIdx.x * kThreads + threadIdx.x;
  if (t >= n) return;
  uint32_t sum = 0;
  for (int e = 0; e < nElements; e++) sum += 4u + elems[e].lens[t];
  chainLens[t] = sum - 4u;
}

// One CTA per tile (persistent).  The record is written as aligned 32-bit words.  Shared memory holds the tile's segment
// table: segment e is element e's [len] field followed by its payload, starting at record offset segStart[e].  Word i
// belongs to the segment its first byte lies in; a word that lies wholly inside a payload is one funnel-shifted load
// from the source arena (whose alignment is arbitrary), a word across a segment boundary is put together byte by byte.
__global__ void __launch_bounds__(kThreads) record_pack_multi_kernel(const RecordElement* elems, int nElements, const int32_t* tileIndex,
                                                                     int firstTileIndex, int n, const uint64_t* crcOff,
                                                                     const uint32_t* crcLen, uint8_t* records) {
  __shared__ uint32_t segStart[G4_MAX_ELEMENTS + 1];  // [nElements] = end of the chain
  __shared__ uint32_t segLen[G4_MAX_ELEMENTS];
  __shared__ const uint8_t* segSrc[G4_MAX_ELEMENTS];
  const int E = nElements;
  for (int t = blockIdx.x; t < n; t += gridDim.x) {
    if (threadIdx.x < E) {
      const RecordElement el = elems[threadIdx.x];
      segLen[threadIdx.x] = el.lens[t];
      segSrc[threadIdx.x] = el.arena + el.offsets[t];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t p = 12;
      for (int e = 0; e < E; e++) {
        segStart[e] = p;
        p += 4u + segLen[e];
      }
      segStart[E] = p;
    }
    __syncthreads();
    uint32_t* w = reinterpret_cast<uint32_t*>(records + crcOff[t]);
    const uint32_t size = crcLen[t] + 4u;
    if (threadIdx.x == 0) {
      w[0] = size;
      w[1] = 2u;  // RecordType.Tile, three reserved zero bytes
      w[2] = uint32_t(tileIndex ? tileIndex[t] : firstTileIndex + t);
    }
    for (int e = 0; e < E; e++) {
      const uint32_t s0 = segStart[e], s1 = segStart[e + 1], p0 = s0 + 4u;
      const uint8_t* src = segSrc[e];
      for (uint32_t i = (s0 + 3u) / 4u + threadIdx.x; i < (s1 + 3u) / 4u; i += kThreads) {
        const uint32_t b = 4u * i;
        uint32_t v = 0;
        if (b >= p0 && b + 4u <= s1) {
          v = load_u32_funnel(src + (b - p0));
        } else {
          int k = e;
          for (uint32_t j = 0; j < 4; j++) {
            const uint32_t q = b + j;
            while (k < E && q >= segStart[k + 1]) k++;
            if (k == E) break;  // past the chain: padding
            const uint32_t r = q - segStart[k];
            const uint32_t byte = r < 4u ? (segLen[k] >> (8u * r)) & 0xffu : segSrc[k][r - 4u];
            v |= byte << (8u * j);
          }
        }
        w[i] = v;
      }
    }
    // zero padding and a zero checksum field (crc32c_kernel fills it in when checksums are enabled)
    for (uint32_t i = (segStart[E] + 3u) / 4u + threadIdx.x; i < size / 4u; i += kThreads) w[i] = 0u;
    __syncthreads();  // the segment table is rewritten for the next tile
  }
}

// One thread per tile: the checks of record_unpack_kernel, then the [len] chain of the nElements elements, which has to
// end at or before the checksum field.  payloadOff / lens are element-major (element e of tile t at e * n + t); a tile
// whose status is not G4_OK gets 0 / 0 for every element.
__global__ void __launch_bounds__(kThreads) record_unpack_multi_kernel(const uint8_t* image, uint64_t imageLen, const uint64_t* contentPos,
                                                                       int n, int nElements, uint64_t* payloadOff, uint32_t* lens,
                                                                       uint64_t* crcOff, uint32_t* crcLen, uint32_t* storedCrc,
                                                                       int32_t* status) {
  const int t = blockIdx.x * kThreads + threadIdx.x;
  if (t >= n) return;
  const uint64_t cp = contentPos[t];
  int st = G4_OK;
  uint32_t cl = 0, sc = 0;
  uint64_t co = 0;
  if (cp == 0) st = G4_DECLINED;  // tile not present in the file
  else if ((cp & 7) || cp < 8 || cp + 8 > imageLen) st = G4_ERR_FORMAT;
  else {
    const uint32_t* h = reinterpret_cast<const uint32_t*>(image + cp - 8);
    const uint32_t size = h[0];
    const uint32_t type = h[1] & 0xffu;
    if (type != 2u || size < 24u || (size & 7u) || cp - 8 + size > imageLen) st = G4_ERR_FORMAT;
    else {
      const uint64_t limit = cp - 8 + size - 4;  // the checksum field
      uint64_t q = cp + 4;                       // element 0's [len]
      for (int e = 0; e < nElements; e++) {
        if (q + 4 > limit) { st = G4_ERR_FORMAT; break; }
        const uint32_t ln = load_u32_funnel(image + q);
        if ((ln >> 31) || q + 4 + ln > limit) { st = G4_ERR_FORMAT; break; }
        payloadOff[size_t(e) * n + t] = q + 4;
        lens[size_t(e) * n + t] = ln;
        q += 4ull + ln;
      }
      if (st == G4_OK) {
        co = cp - 8;
        cl = size - 4u;
        sc = *reinterpret_cast<const uint32_t*>(image + limit);
      }
    }
  }
  if (st != G4_OK) {
    for (int e = 0; e < nElements; e++) {
      payloadOff[size_t(e) * n + t] = 0;
      lens[size_t(e) * n + t] = 0;
    }
  }
  crcOff[t] = co;
  crcLen[t] = cl;
  storedCrc[t] = sc;
  status[t] = st;
}

__global__ void __launch_bounds__(kThreads) record_verify_multi_kernel(const uint32_t* computed, const uint32_t* stored, int n,
                                                                       int nElements, uint64_t* payloadOff, uint32_t* lens,
                                                                       int32_t* status) {
  const int t = blockIdx.x * kThreads + threadIdx.x;
  if (t >= n) return;
  if (status[t] != G4_OK || computed[t] == stored[t]) return;
  status[t] = G4_CHECKSUM_MISMATCH;
  for (int e = 0; e < nElements; e++) {
    payloadOff[size_t(e) * n + t] = 0;
    lens[size_t(e) * n + t] = 0;
  }
}

cudaError_t launch_record_chain_lens(const RecordElement* elems, int nElements, int n, uint32_t* chainLens, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  record_chain_lens_kernel<<<(n + kThreads - 1) / kThreads, kThreads, 0, s>>>(elems, nElements, n, chainLens);
  return cudaGetLastError();
}
cudaError_t launch_record_pack_multi(const RecordElement* elems, int nElements, const int32_t* tileIndex, int firstTileIndex, int n,
                                     const uint64_t* crcOff, const uint32_t* crcLen, uint8_t* records, int nCtas, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  record_pack_multi_kernel<<<nCtas, kThreads, 0, s>>>(elems, nElements, tileIndex, firstTileIndex, n, crcOff, crcLen, records);
  return cudaGetLastError();
}
cudaError_t launch_record_unpack_multi(const uint8_t* image, uint64_t imageLen, const uint64_t* contentPos, int n, int nElements,
                                       uint64_t* payloadOff, uint32_t* lens, uint64_t* crcOff, uint32_t* crcLen, uint32_t* storedCrc,
                                       int32_t* status, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  record_unpack_multi_kernel<<<(n + kThreads - 1) / kThreads, kThreads, 0, s>>>(image, imageLen, contentPos, n, nElements, payloadOff, lens,
                                                                               crcOff, crcLen, storedCrc, status);
  return cudaGetLastError();
}
cudaError_t launch_record_verify_multi(const uint32_t* computed, const uint32_t* stored, int n, int nElements, uint64_t* payloadOff,
                                       uint32_t* lens, int32_t* status, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  record_verify_multi_kernel<<<(n + kThreads - 1) / kThreads, kThreads, 0, s>>>(computed, stored, n, nElements, payloadOff, lens, status);
  return cudaGetLastError();
}

cudaError_t launch_crc32c(const uint8_t* data, const uint64_t* offsets, const uint32_t* sizes, int n, uint32_t* out, int storeAtEnd,
                          cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  const int perCta = kCrcThreads / 32;
  crc32c_kernel<<<(n + perCta - 1) / perCta, kCrcThreads, 0, s>>>(data, offsets, sizes, n, out, storeAtEnd);
  return cudaGetLastError();
}
cudaError_t launch_record_layout(const uint32_t* lens, int n, uint64_t basePos, uint64_t* contentPos, uint64_t* crcOff, uint32_t* crcLen,
                                 uint64_t* total, cudaStream_t s) {
  record_layout_kernel<<<1, kThreads, 0, s>>>(lens, n, basePos, contentPos, crcOff, crcLen, total);
  return cudaGetLastError();
}
cudaError_t launch_record_pack(const uint8_t* arena, const uint64_t* offsets, const uint32_t* lens, const int32_t* tileIndex,
                               int firstTileIndex, int n, const uint64_t* crcOff, const uint32_t* crcLen, uint8_t* records, int nCtas,
                               cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  record_pack_kernel<<<nCtas, kThreads, 0, s>>>(arena, offsets, lens, tileIndex, firstTileIndex, n, crcOff, crcLen, records);
  return cudaGetLastError();
}
cudaError_t launch_record_unpack(const uint8_t* image, uint64_t imageLen, const uint64_t* contentPos, int n, uint64_t* payloadOff,
                                 uint32_t* lens, uint64_t* crcOff, uint32_t* crcLen, uint32_t* storedCrc, int32_t* status, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  record_unpack_kernel<<<(n + kThreads - 1) / kThreads, kThreads, 0, s>>>(image, imageLen, contentPos, n, payloadOff, lens, crcOff, crcLen,
                                                                         storedCrc, status);
  return cudaGetLastError();
}
cudaError_t launch_record_verify(const uint32_t* computed, const uint32_t* stored, int n, int32_t* status, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  record_verify_kernel<<<(n + kThreads - 1) / kThreads, kThreads, 0, s>>>(computed, stored, n, status);
  return cudaGetLastError();
}

}  // namespace g4
