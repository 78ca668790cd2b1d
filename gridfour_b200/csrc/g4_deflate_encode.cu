// g4_deflate_encode.cu -- encode side of CodecDeflate and CodecFloat, and the generic zlib-stream worker kernel.
//
// Reference (under /root/reference/core/src/main/java/org/gridfour/compress/):
//   CodecDeflate.java:157-202 (encode: best of the three predictors by packing length, strict <),
//   CodecDeflate.java:204-228 (compress: Deflater(6), finish(), one deflate() into nM32+128 bytes at offset 10),
//   CodecFloat.java:300-313 (encodeDeltas), :328-392 (encodeFloats), :268-283 (doDeflate: Deflater(9), n+128 bytes)
//
// Every codec that needs zlib streams runs the same four stages:
//   size   one CTA per tile computes the byte length of each stream it will hand to DEFLATE
//   scan   exclusive scan of the padded lengths -> stream offsets (exact-size staging, no 6n worst-case slabs)
//   write  one CTA per tile writes the streams (M32 bytes in predictor stream order / float byte planes)
//   zlib   one THREAD per stream replays zlib's deflate_slow (g4_deflate_enc.cuh); LZ77 hash-chain matching is
//          serial per stream, so the parallelism is across the tens of thousands of streams of a band
//   pick   one CTA per tile selects / assembles the packing in the tile's candidate slot
#include "g4_kernels.h"
#include "g4_device.cuh"
#include "g4_predict.cuh"
#include "g4_m32stream.cuh"
#include "g4_deflate_enc.cuh"
#include "g4_bitpack.cuh"

namespace g4 {

size_t deflate_work_bytes() { return sizeof(DeflateWork); }

// ---- stream offsets -----------------------------------------------------------------------------------------
// inOff[j] = sum_{i<j} align16(inLen[i] + 16); the output slot of stream j starts at inOff[j] + 112*j in the output
// buffer (capacity inLen[j] + 128).  One CTA.
__global__ void __launch_bounds__(kThreads) stream_offsets_kernel(const uint32_t* inLen, uint64_t* inOff, int n, uint64_t* total) {
  __shared__ unsigned long long sm[kWarps];
  __shared__ unsigned long long carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int t0 = 0; t0 < n; t0 += kThreads) {
    int t = t0 + threadIdx.x;
    unsigned long long x = t < n ? ((unsigned long long)(inLen[t]) + 31ull) & ~15ull : 0ull;
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
    if (t < n) inOff[t] = base + inc - x;
    __syncthreads();
    if (threadIdx.x == kThreads - 1) carry = base + inc;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}

// ---- one thread per zlib stream ---------------------------------------------------------------------------------
// General form (any length; the only one for streams longer than kDefStagedMax).  With a.bigOnly set it leaves the
// short streams to the staged kernels below.
__global__ void __launch_bounds__(32) deflate_streams_kernel(StreamArgs a) {
  DeflateWork* W = static_cast<DeflateWork*>(a.work) + (size_t(blockIdx.x) * blockDim.x + threadIdx.x);
  for (;;) {
    const int j = atomicAdd(a.counter, 1);
    if (j >= a.nStreams) break;
    const uint32_t n = a.inLen[j];
    if (a.bigOnly && n <= kDefStagedMax) continue;
    if (n == 0) { a.outLen[j] = 0; continue; }  // stream not produced (tile declined by the size stage)
    const uint64_t off = a.inOff[j];
    a.outLen[j] = deflate_stream(a.inBuf + off, n, a.outBuf + off + 112ull * uint64_t(j), n + uint32_t(a.capExtra), W, a.level);
  }
}

// ---- staged form for streams of at most kDefStagedMax bytes (g4_deflate_enc.cuh, "Staged form") ------------------------
// sort: one 128-thread CTA per stream, bucket cursors (32768 x uint16 = 64 KB) in shared memory.
//   pass 1 (all threads)  hash of every position, parked in a scratch array; bucket counts by shared-memory atomics,
//   scan   (all threads)  counts -> bucket starts,
//   pass 2 (warp 0)       slots in stream order: positions are taken 32 at a time; __match_any_sync groups the lanes
//                         of a chunk by hash, a position's slot is (bucket cursor) + (lanes below it with the same
//                         hash) and the highest lane of every group advances the cursor by the group's size.  Eight
//                         chunks of hashes are loaded and grouped ahead of the serial cursor updates.
// The list alone is the result: a slot's bucket and its place in it are read off the (hash, position) order by the match
// kernel, so no rank array is written (the scattered 2-byte stores are what this kernel's time is made of).
// (Tried and dropped: per-position shared-memory atomics instead of the grouped update, with a fix-up of the order
// inside a chunk -- the two extra passes over HBM cost more than the grouping, 64 ms instead of 41 ms.)
constexpr int kSortThreads = 128;
__global__ void __launch_bounds__(kSortThreads) deflate_sort_kernel(StagedArgs a) {
  extern __shared__ uint16_t sortTab[];
  __shared__ uint32_t warpSum[kSortThreads / 32];
  __shared__ int sj;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t ltMask = (1u << lane) - 1u;
  uint32_t* t32 = reinterpret_cast<uint32_t*>(sortTab);
  for (;;) {
    __syncthreads();
    if (tid == 0) sj = a.jBegin + atomicAdd(a.counters + 0, 1);
    __syncthreads();
    const int j = sj;
    if (j >= a.jEnd) break;
    const uint32_t n = a.inLen[j];
    if (n < 3 || n > kDefStagedMax) continue;
    const uint64_t off = a.inOff[j];
    const uint8_t* in = a.inBuf + off;
    uint16_t* sorted = a.sorted + (off - a.baseOff);
    uint16_t* hashOf = reinterpret_cast<uint16_t*>(a.tableQ + (off - a.baseOff));  // the match tables are not written yet
    uint16_t* slotOf = a.lazy ? a.rank + (off - a.baseOff) : nullptr;
    const uint32_t nPos = n - 2;
    {
      uint4* t4 = reinterpret_cast<uint4*>(sortTab);
      for (int i = tid; i < kDefWSize * 2 / 16; i += kSortThreads) t4[i] = make_uint4(0, 0, 0, 0);
    }
    __syncthreads();
    {  // four positions per thread and step from two aligned words (the stream starts 16-byte aligned and is zero-padded)
      const uint32_t* in32 = reinterpret_cast<const uint32_t*>(in);
      uint2* hash4 = reinterpret_cast<uint2*>(hashOf);
#pragma unroll 4
      for (uint32_t g = tid; g * 4u < nPos; g += kSortThreads) {
        const uint32_t w0 = __ldg(in32 + g), w1 = __ldg(in32 + g + 1);
        uint32_t hh[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const uint32_t x = i ? __funnelshift_r(w0, w1, 8u * uint32_t(i)) : w0;
          hh[i] = (((x & 0xffu) << 10) ^ (((x >> 8) & 0xffu) << 5) ^ ((x >> 16) & 0xffu)) & uint32_t(kDefHashMask);
          if (g * 4u + uint32_t(i) < nPos) atomicAdd(&t32[hh[i] >> 1], (hh[i] & 1u) ? 0x10000u : 1u);
        }
        hash4[g] = make_uint2(hh[0] | (hh[1] << 16), hh[2] | (hh[3] << 16));
      }
    }
    __syncthreads();
    {  // exclusive scan of the 32768 counts: every warp scans a quarter (two counts per lane and step), then the
       // quarters are offset by the sums of the quarters before them
      const int q0 = warp * (kDefWSize / 2 / 4);
      uint32_t carry = 0;
      for (int i0 = 0; i0 < kDefWSize / 2 / 4; i0 += 32) {
        const uint32_t v = t32[q0 + i0 + lane];
        const uint32_t c0 = v & 0xffffu, c1 = v >> 16;
        uint32_t inc = c0 + c1;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
          if (lane >= d) inc += y;
        }
        const uint32_t ex = carry + inc - (c0 + c1);
        t32[q0 + i0 + lane] = (ex & 0xffffu) | ((ex + c0) << 16);
        carry += __shfl_sync(0xffffffffu, inc, 31);
      }
      if (lane == 0) warpSum[warp] = carry;
      __syncthreads();
      uint32_t add = 0;
      for (int w = 0; w < warp; w++) add += warpSum[w];
      if (add) {
        const uint32_t add2 = add | (add << 16);  // no carry between the halves: every start is < 65536
        for (int i0 = 0; i0 < kDefWSize / 2 / 4; i0 += 32) t32[q0 + i0 + lane] += add2;
      }
    }
    __syncthreads();
    if (warp == 0) {
      uint32_t hN[8];
#pragma unroll
      for (int c = 0; c < 8; c++) {
        const uint32_t p = uint32_t(c) * 32u + uint32_t(lane);
        hN[c] = p < nPos ? uint32_t(hashOf[p]) : (0x10000u | uint32_t(lane));
      }
      for (uint32_t base = 0; base < nPos; base += 256) {
        uint32_t h[8], mm[8];
#pragma unroll
        for (int c = 0; c < 8; c++) h[c] = hN[c];
#pragma unroll
        for (int c = 0; c < 8; c++) {  // next group's hashes: in flight during this group's serial part
          const uint32_t p = base + 256u + uint32_t(c) * 32u + uint32_t(lane);
          hN[c] = p < nPos ? uint32_t(hashOf[p]) : (0x10000u | uint32_t(lane));
        }
#pragma unroll
        for (int c = 0; c < 8; c++) mm[c] = __match_any_sync(0xffffffffu, h[c]);
#pragma unroll
        for (int c = 0; c < 8; c++) {
          const uint32_t m = mm[c];
          if (h[c] < 0x10000u) {
            const uint32_t cur = sortTab[h[c]];
            const uint32_t slot = cur + uint32_t(__popc(m & ltMask));
            sorted[slot] = uint16_t(base + uint32_t(c) * 32u + uint32_t(lane));
            if (slotOf) slotOf[base + uint32_t(c) * 32u + uint32_t(lane)] = uint16_t(slot);
            if ((m >> lane) == 1u) sortTab[h[c]] = uint16_t(cur + __popc(m));
          }
          __syncwarp();
        }
      }
    }
  }
}

// match: the chain of the position in slot i is slots i-1, i-2, ... of the sorted list,
// so the candidates of NEIGHBOURING slots are one sliding window.  The CTA keeps, for a window of slots, the position and
// the 8 bytes that start there (one 64-bit key); a thread compares its key with the keys behind it: XOR + mask test per
// candidate, no byte loads and no data-dependent inner loop.  The common prefix of two positions is exact from the keys
// while it is shorter than 8; equal keys (prefix >= 8) go on comparing the stream itself.  zlib's candidate filter
// (match[best_len] == scan_end ...) is the statement "common prefix > best_len", which is what the mask test decides.
// The distance rules (MAX_DIST, position 0 = NIL) cut the chain at a candidate count that is found before the walk
// (positions fall along the chain: binary search), so the walk itself reads keys only.
// The results are indexed by POSITION while the threads run in slot (= hash) order: written straight to HBM that is one
// scattered 32-byte sector per entry, and DRAM's rate of such writes -- not the matching -- set the kernel's time
// (43 GB written + 76 GB read for 1.4 GB of input, profiles/).  The table of a stream (4 bytes per position) therefore
// fills in shared memory and leaves with coalesced stores; streams too long for that keep the scattered store.
// kMatchChain = chain length of the levels below 9 (slots that must stay behind a round; level 9 takes deflate_lazy_kernel),
// SB = slots per round, tabCap = entries of the shared-memory table.
// GROUPS: the CTA works as that many independent thread groups, each with its own window, taking the rounds of a stream
// in turn and synchronising with a named barrier of its own: while one group waits for the gathers that fill its window,
// the other walks (with one 205 KB CTA per SM there is no second CTA to do that).
constexpr int kMatchChain = 128;
template <int SB, int GROUPS, int NT_MAX, int MIN_CTAS>
__global__ void __launch_bounds__(NT_MAX, MIN_CTAS) deflate_match_window_kernel(StagedArgs a, uint32_t tabCap) {
  extern __shared__ __align__(16) unsigned char matchSm[];
  const uint32_t nThr = blockDim.x / GROUPS, grp = threadIdx.x / nThr, tid = threadIdx.x - grp * nThr;
  unsigned char* winSm = matchSm + size_t(grp) * (size_t(kMatchChain + SB) * 16);
  uint2* keyS = reinterpret_cast<uint2*>(winSm);
  uint32_t* filtS = reinterpret_cast<uint32_t*>(winSm + size_t(kMatchChain + SB) * 8);
  uint32_t* hpS = reinterpret_cast<uint32_t*>(winSm + size_t(kMatchChain + SB) * 12);  // hash << 16 | position: rises with the slot
  uint32_t* tabS = reinterpret_cast<uint32_t*>(matchSm + size_t(GROUPS) * size_t(kMatchChain + SB) * 16);
  __shared__ int sj;
  auto group_sync = [&]() {
    if (GROUPS == 1) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(1u + grp), "r"(nThr) : "memory");
  };
  const DeflateLevel L = deflate_level(a.level);
  const uint32_t maxChain = uint32_t(L.maxChain) < uint32_t(kMatchChain) ? uint32_t(L.maxChain) : uint32_t(kMatchChain);
  const uint32_t quarter = uint32_t(L.maxChain) >> 2;
  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) sj = a.jBegin + atomicAdd(a.counters + 1, 1);
    __syncthreads();
    const int j = sj;
    if (j >= a.jEnd) break;
    const uint32_t n = a.inLen[j];
    if (n < 3 || n > kDefStagedMax) continue;
    const uint64_t off = a.inOff[j];
    const uint8_t* in = a.inBuf + off;
    const uint16_t* sorted = a.sorted + (off - a.baseOff);
    uint32_t* table = a.table + (off - a.baseOff);
    uint32_t* tableQ = a.tableQ + (off - a.baseOff);
    const uint32_t nPos = n - 2;
    const bool inSm = nPos <= tabCap;
    for (uint32_t base = grp * uint32_t(SB); base < nPos; base += uint32_t(GROUPS) * uint32_t(SB)) {
      const uint32_t end = base + SB < nPos ? base + SB : nPos;
      // window = slots [first, end), index = slot + kMatchChain - base
      const uint32_t first = base >= uint32_t(kMatchChain) ? base - uint32_t(kMatchChain) : 0u;
      group_sync();
      for (uint32_t s = first + tid; s < end; s += nThr) {
        const uint32_t p = sorted[s];
        const uintptr_t ad = reinterpret_cast<uintptr_t>(in + p);
        const uint32_t* q = reinterpret_cast<const uint32_t*>(ad & ~uintptr_t(3));
        const uint32_t sh = uint32_t(ad & 3u) * 8u;
        const uint32_t w0 = q[0], w1 = q[1], w2 = q[2];  // in[] is padded with 16 zero bytes past n
        const uint32_t kl = __funnelshift_r(w0, w1, sh), kh = __funnelshift_r(w1, w2, sh);
        hpS[s + kMatchChain - base] = (((((kl & 0xffu) << 10) ^ (((kl >> 8) & 0xffu) << 5) ^ ((kl >> 16) & 0xffu)) & uint32_t(kDefHashMask)) << 16) | p;
        keyS[s + kMatchChain - base] = make_uint2(kl, kh);
        // 32-bit filter word.  Inside a hash bucket, byte 1 fixes byte 2 and the low five bits of byte 0 (the hash is
        // b0 << 10 ^ b1 << 5 ^ b2, 15 bits), so {b0 >> 5, b1} is the whole 3-byte prefix; then bytes 3, 4 and five bits
        // of byte 5.  Fields in byte order: a mask over the low bits tests "at least that many bytes in common".
        filtS[s + kMatchChain - base] = ((kl >> 5) & 7u) | (((kl >> 8) & 0xffu) << 3) | ((kl >> 24) << 11) | ((kh & 0xffu) << 19) | (((kh >> 8) & 31u) << 27);
      }
      group_sync();
      for (uint32_t slot = base + tid; slot < end; slot += nThr) {
        const uint32_t li = slot + kMatchChain - base;
        const uint2 my = keyS[li];
        const uint32_t hp = hpS[li];
        const uint32_t p = hp & 0xffffu;
        const uint32_t lookahead = n - p;
        const int maxLen = lookahead < uint32_t(kDefMaxMatch) ? int(lookahead) : kDefMaxMatch;
        const int niceMatch = uint32_t(L.niceLength) > lookahead ? int(lookahead) : L.niceLength;
        // Candidates: the slots behind this one that hold the same hash and a position above `limit` (nearer than
        // MAX_DIST; position 0 doubles as NIL), at most maxChain of them.  (hash, position) rises with the slot, so they
        // are the run that ends here: lower bound by binary search.  zlib's first candidate may sit at MAX_DIST exactly.
        const uint32_t limit = p > uint32_t(kDefMaxDist) ? p - uint32_t(kDefMaxDist) : 0u;
        const uint32_t want = (hp & 0xffff0000u) | (limit + 1u);
        uint32_t nCand = slot < maxChain ? slot : maxChain;
        if (nCand && hpS[li - nCand] < want) {
          uint32_t lo = 0, hi = nCand;  // entry(lo) >= want (lo = 0: the slot itself), entry(hi) < want
          while (hi - lo > 1u) {
            const uint32_t mid = (lo + hi) >> 1;
            if (hpS[li - mid] >= want) lo = mid; else hi = mid;
          }
          nCand = (lo == 0u && limit != 0u && hpS[li - 1] == want - 1u) ? 1u : lo;
        }
        int bestLen = kDefMinMatch - 1;
        uint32_t bestDist = p;
        uint32_t mLo = 0x00ffffffu, mHi = 0u;  // bytes 0 .. bestLen of the key
        const uint32_t myF = filtS[li];
        uint32_t mF = 0x7ffu;  // the same bytes in the filter word (a necessary condition once bestLen reaches 5)
        bool done = false;
        // one candidate, exactly: true when the walk is over (nice match)
        auto exact = [&](uint32_t k) -> bool {
          const uint2 ck = keyS[li - k];
          const uint32_t xl = ck.x ^ my.x, xh = ck.y ^ my.y;
          if (((xl & mLo) | (xh & mHi)) != 0u) return false;
          const uint32_t cur = hpS[li - k] & 0xffffu;
          int len;
          if (xl) len = (__ffs(int(xl)) - 1) >> 3;
          else if (xh) len = 4 + ((__ffs(int(xh)) - 1) >> 3);
          else {
            len = 8;
            const uint8_t* scan = in + p;
            const uint8_t* match = in + cur;
            if (bestLen >= 8 && (match[bestLen] != scan[bestLen] || match[bestLen - 1] != scan[bestLen - 1])) return false;
            bool differ = false;
            while (len + 4 <= maxLen) {
              const uint32_t x = def_load32(scan + len) ^ def_load32(match + len);
              if (x) { len += (__ffs(int(x)) - 1) >> 3; differ = true; break; }
              len += 4;
            }
            if (!differ)
              while (len < maxLen && scan[len] == match[len]) len++;
          }
          if (len > maxLen) len = maxLen;
          if (len > bestLen) {
            bestLen = len;
            bestDist = p - cur;
            if (len >= niceMatch) { done = true; return true; }
            const uint32_t nb8 = uint32_t(len + 1) * 8u;  // bits of the key that a better candidate must share
            const unsigned long long m64 = nb8 >= 64u ? ~0ull : (1ull << nb8) - 1ull;
            mLo = uint32_t(m64);
            mHi = uint32_t(m64 >> 32);
            const uint32_t fb = uint32_t(len) * 8u - 5u;  // 11 + 8 (len - 2) filter bits
            mF = fb >= 32u ? 0xffffffffu : (1u << fb) - 1u;
          }
          return false;
        };
        // The walk: the first candidates one at a time (every lane of the warp finds its first matches there), then
        // blocks of up to 32 candidates: a scan over the filter words (one 32-bit load and two logic operations per
        // candidate, no branch) marks the candidates that may share more than bestLen bytes, and the marked ones are
        // then taken nearest first on the 64-bit keys -- all lanes of the warp together, instead of every lane
        // stopping the warp's scan for its own candidate.  (The mark uses bestLen of the block's start: a superset.)
        auto walk = [&](uint32_t k0, uint32_t k1) {
          uint32_t k = k0;
          for (; k <= k1 && k < k0 + 4u; k++)
            if (exact(k)) return;
          while (k <= k1) {
            const uint32_t left = k1 - k + 1u;
            uint32_t pend = 0;
            if (left >= 32u) {
#pragma unroll
              for (uint32_t q = 0; q < 32u; q += 4u) {
                const uint32_t f0 = filtS[li - k - q], f1 = filtS[li - k - q - 1u], f2 = filtS[li - k - q - 2u], f3 = filtS[li - k - q - 3u];
                if (((f0 ^ myF) & mF) == 0u) pend |= 1u << q;
                if (((f1 ^ myF) & mF) == 0u) pend |= 2u << q;
                if (((f2 ^ myF) & mF) == 0u) pend |= 4u << q;
                if (((f3 ^ myF) & mF) == 0u) pend |= 8u << q;
              }
            } else {
              uint32_t q = 0;
              for (; q + 4u <= left; q += 4u) {
                const uint32_t f0 = filtS[li - k - q], f1 = filtS[li - k - q - 1u], f2 = filtS[li - k - q - 2u], f3 = filtS[li - k - q - 3u];
                uint32_t hit = 0;
                if (((f0 ^ myF) & mF) == 0u) hit |= 1u;
                if (((f1 ^ myF) & mF) == 0u) hit |= 2u;
                if (((f2 ^ myF) & mF) == 0u) hit |= 4u;
                if (((f3 ^ myF) & mF) == 0u) hit |= 8u;
                pend |= hit << q;
              }
              for (; q < left; q++)
                if (((filtS[li - k - q] ^ myF) & mF) == 0u) pend |= 1u << q;
            }
            while (pend) {
              const uint32_t q = uint32_t(__ffs(int(pend))) - 1u;
              pend &= pend - 1u;
              if (exact(k + q)) return;
            }
            k += left >= 32u ? 32u : left;
          }
        };
        walk(1u, nCand < quarter ? nCand : quarter);
        const uint32_t quarterEntry = def_pack_match(bestLen, bestDist);  // = the full result when the chain ends here
        if (!done && nCand > quarter) walk(quarter + 1u, nCand);
        uint32_t full = def_pack_match(bestLen, bestDist);
        if (full != quarterEntry) { tableQ[p] = quarterEntry; full |= 0x80000000u; }  // rare: the scattered store stays
        if (inSm) tabS[p] = full; else table[p] = full;
      }
    }
    if (inSm) {
      __syncthreads();
      uint4* dst = reinterpret_cast<uint4*>(table);  // 64-byte aligned: stream offsets are multiples of 16 positions
      const uint4* src = reinterpret_cast<const uint4*>(tabS);
      for (uint32_t i = threadIdx.x; i < (nPos + 3u) / 4u; i += blockDim.x) dst[i] = src[i];
    }
  }
}

// lazy (deep levels, CodecFloat's Deflater(9)): with 4096-candidate chains the table of EVERY position costs a hundred
// times what zlib spends, because zlib never searches the positions a match covers -- and the float planes are mostly
// long matches.  Here ONE WARP per stream runs deflate_slow itself and searches only where zlib does; the search is what
// the warp shares: 32 candidates of the chain (consecutive slots behind the position's slot in the sorted list) per
// step, each lane one candidate -- distance rules, bucket membership (hash of the candidate's bytes), common prefix from
// two 64-bit keys and then the stream itself -- and a warp reduction picks the longest, nearest first, exactly
// longest_match()'s answer (a later candidate replaces the best only when strictly longer; the walk ends at nice_match,
// at the chain length, at the first candidate beyond MAX_DIST or outside the bucket).
__global__ void __launch_bounds__(128, 12) deflate_lazy_kernel(StagedArgs a) {
  const uint32_t lane = threadIdx.x & 31u;
  const DeflateLevel L = deflate_level(a.level);
  for (;;) {
    int j = 0;
    if (lane == 0) j = a.jBegin + atomicAdd(a.counters + 1, 1);
    j = __shfl_sync(0xffffffffu, j, 0);
    if (j >= a.jEnd) break;
    const uint32_t n = a.inLen[j];
    if (n == 0 || n > kDefStagedMax) continue;
    const uint64_t off = a.inOff[j];
    const uint8_t* in = a.inBuf + off;
    const uint32_t* in32 = reinterpret_cast<const uint32_t*>(in);
    const uint16_t* sorted = a.sorted + (off - a.baseOff);
    const uint16_t* slotOf = a.rank + (off - a.baseOff);
    uint16_t* symDist = reinterpret_cast<uint16_t*>(a.table + (off - a.baseOff));
    uint8_t* symLc = reinterpret_cast<uint8_t*>(a.tableQ + (off - a.baseOff));
    DeflateBlocks* B = a.blocks + (j - a.jBegin);
    auto key_at = [&](uint32_t p, uint32_t& lo, uint32_t& hi) {
      const uint32_t* q = in32 + (p >> 2);
      const uint32_t sh = (p & 3u) * 8u;
      const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2);
      lo = __funnelshift_r(w0, w1, sh);
      hi = __funnelshift_r(w1, w2, sh);
    };
    uint32_t strstart = 0, matchStart = 0, prevMatch = 0, k = 0, inBlock = 0, nBlocks = 0;
    int matchLength = kDefMinMatch - 1, prevLength = kDefMinMatch - 1;
    bool matchAvailable = false;
    auto tally = [&](uint32_t dist, uint32_t lc) -> bool {
      if (lane == 0) { symDist[k] = uint16_t(dist); symLc[k] = uint8_t(lc); }
      k++;
      return ++inBlock == uint32_t(kDefLitBufSize - 1);
    };
    auto flush = [&]() {
      if (lane == 0) { B->symEnd[nBlocks] = k; B->posEnd[nBlocks] = strstart; }
      nBlocks++;
      inBlock = 0;
    };
    while (strstart < n) {
      const uint32_t p = strstart;
      const uint32_t lookahead = n - p;
      prevLength = matchLength;
      prevMatch = matchStart;
      matchLength = kDefMinMatch - 1;
      if (lookahead >= uint32_t(kDefMinMatch) && prevLength < L.maxLazy) {
        const uint32_t slot = slotOf[p];
        const uint32_t chain = prevLength >= L.goodLength ? uint32_t(L.maxChain) >> 2 : uint32_t(L.maxChain);
        const uint32_t nMax = slot < chain ? slot : chain;
        const int maxLen = lookahead < uint32_t(kDefMaxMatch) ? int(lookahead) : kDefMaxMatch;
        const int niceMatch = uint32_t(L.niceLength) > lookahead ? int(lookahead) : L.niceLength;
        const uint32_t limit = p > uint32_t(kDefMaxDist) ? p - uint32_t(kDefMaxDist) : 0u;
        uint32_t klo, khi;
        key_at(p, klo, khi);
        int bestLen = prevLength;
        uint32_t bestStart = 0;
        uint32_t curNext = lane + 1u <= nMax ? uint32_t(sorted[slot - lane - 1u]) : 0u;
        for (uint32_t k0 = 0; k0 < nMax; k0 += 32u) {
          const uint32_t kk = k0 + lane + 1u;
          bool valid = kk <= nMax;
          uint32_t cur = curNext, clo = 0, chi = 0;
          if (kk + 32u <= nMax) curNext = sorted[slot - kk - 32u];  // the next step's candidate: in flight during this one
          if (valid) valid = kk == 1u ? !(cur == 0u || p - cur > uint32_t(kDefMaxDist)) : cur > limit;
          if (valid) {
            key_at(cur, clo, chi);
            valid = ((clo ^ klo) & 0x00ffffffu) == 0u ||
                    ((((clo & 0xffu) << 10) ^ (((clo >> 8) & 0xffu) << 5) ^ ((clo >> 16) & 0xffu)) & uint32_t(kDefHashMask)) ==
                        ((((klo & 0xffu) << 10) ^ (((klo >> 8) & 0xffu) << 5) ^ ((klo >> 16) & 0xffu)) & uint32_t(kDefHashMask));
          }
          const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
          const uint32_t nv = vmask == 0xffffffffu ? 32u : uint32_t(__ffs(int(~vmask))) - 1u;  // the chain ends at the first invalid candidate
          int len = 0;
          if (lane < nv) {
            const uint32_t xl = clo ^ klo, xh = chi ^ khi;
            if (xl) len = (__ffs(int(xl)) - 1) >> 3;
            else if (xh) len = 4 + ((__ffs(int(xh)) - 1) >> 3);
            else {
              len = 8;
              const uint8_t* scan = in + p;
              const uint8_t* match = in + cur;
              if (bestLen >= 8 && (match[bestLen] != scan[bestLen] || match[bestLen - 1] != scan[bestLen - 1])) len = 0;
              else {
                bool differ = false;
                while (len + 4 <= maxLen) {
                  const uint32_t x = def_load32(scan + len) ^ def_load32(match + len);
                  if (x) { len += (__ffs(int(x)) - 1) >> 3; differ = true; break; }
                  len += 4;
                }
                if (!differ)
                  while (len < maxLen && scan[len] == match[len]) len++;
              }
            }
            if (len > maxLen) len = maxLen;
          }
          const int stepMax = __reduce_max_sync(0xffffffffu, len);
          if (stepMax > bestLen) {
            const uint32_t who = uint32_t(__ffs(int(__ballot_sync(0xffffffffu, len == stepMax)))) - 1u;  // nearest of the longest
            bestLen = stepMax;
            bestStart = __shfl_sync(0xffffffffu, cur, int(who));
            if (bestLen >= niceMatch) break;
          }
          if (nv < 32u) break;
        }
        if (bestLen > prevLength) {
          matchLength = bestLen;
          matchStart = bestStart;
          if (matchLength == kDefMinMatch && strstart - matchStart > uint32_t(kDefTooFar)) matchLength = kDefMinMatch - 1;
        }
      }
      if (prevLength >= kDefMinMatch && matchLength <= prevLength) {
        const bool bflush = tally(strstart - 1 - prevMatch, uint32_t(prevLength - kDefMinMatch));
        strstart += uint32_t(prevLength - 1);
        matchAvailable = false;
        matchLength = kDefMinMatch - 1;
        if (bflush) flush();
      } else if (matchAvailable) {
        const bool bflush = tally(0, in[strstart - 1]);
        if (bflush) flush();
        strstart++;
      } else {
        matchAvailable = true;
        strstart++;
      }
    }
    if (matchAvailable) tally(0, in[strstart - 1]);
    flush();
    if (lane == 0) B->nBlocks = nBlocks;
  }
}

// decide: one THREAD per stream runs the table-driven lazy loop (deflate_decide_table in g4_deflate_enc.cuh is the host
// form) and leaves the symbol list in the (now dead) sorted / rank arrays of the stream.  The table entries and the input bytes of a
// stream come through a per-thread shared-memory ring filled by cp.async (16 positions per chunk, kDecRing chunks in
// flight), so that a step of the lazy loop costs a shared-memory read instead of a DRAM round trip that the 31 other
// lanes of the warp wait for as well.
constexpr int kDecChunk = 16, kDecRing = 4, kDecRow = kDecChunk * kDecRing;  // chunk: 16 entries = 64 bytes + 16 input bytes
// One stream per lane of a one-warp CTA (fewer streams per warp measured slower, DESIGN.md 6.1.1).
__global__ void __launch_bounds__(32) deflate_decide_ring_kernel(StagedArgs a) {
  __shared__ __align__(16) uint32_t tabS[32][kDecRow + 4];  // +4 entries: rows 16 bytes apart in the banks
  __shared__ __align__(16) uint8_t byteS[32][kDecRow + 16];
  // symbols leave 16 bytes at a time (8 distances / 16 length-or-literal bytes): a warp's scalar stores are 32 L2
  // transactions each, and at two per step they, not the loop, set the kernel's time
  __shared__ __align__(16) uint16_t distS[32][8 + 8];
  __shared__ __align__(16) uint8_t lcS[32][16 + 16];
  const int lane = threadIdx.x;
  const DeflateLevel L = deflate_level(a.level);
  const uint32_t tabBase = uint32_t(__cvta_generic_to_shared(&tabS[lane][0]));
  const uint32_t byteBase = uint32_t(__cvta_generic_to_shared(&byteS[lane][0]));
  for (;;) {
    const int j = a.jBegin + atomicAdd(a.counters + 2, 1);
    if (j >= a.jEnd) break;
    const uint32_t n = a.inLen[j];
    if (n == 0 || n > kDefStagedMax) continue;
    const uint64_t off = a.inOff[j];
    const uint8_t* in = a.inBuf + off;
    const uint32_t* table = a.table + (off - a.baseOff);
    const uint32_t* tableQ = a.tableQ + (off - a.baseOff);
    uint16_t* symDist = a.sorted + (off - a.baseOff);
    uint8_t* symLc = reinterpret_cast<uint8_t*>(a.rank + (off - a.baseOff));
    DeflateBlocks* B = a.blocks + (j - a.jBegin);
    const uint32_t nChunks = (n + uint32_t(kDecChunk) - 1u) / uint32_t(kDecChunk);
    uint32_t fetched = 0, curChunk = 0xffffffffu;
    uint32_t strstart = 0, matchStart = 0, prevMatch = 0, k = 0, inBlock = 0, nBlocks = 0;
    int matchLength = kDefMinMatch - 1, prevLength = kDefMinMatch - 1;
    bool matchAvailable = false;
    uint32_t lastByte = 0;
    auto tally = [&](uint32_t dist, uint32_t lc) -> bool {
      distS[lane][k & 7u] = uint16_t(dist);
      lcS[lane][k & 15u] = uint8_t(lc);
      k++;
      if ((k & 7u) == 0u) {
        *reinterpret_cast<uint4*>(symDist + (k - 8u)) = *reinterpret_cast<const uint4*>(&distS[lane][0]);
        if ((k & 15u) == 0u) *reinterpret_cast<uint4*>(symLc + (k - 16u)) = *reinterpret_cast<const uint4*>(&lcS[lane][0]);
      }
      return ++inBlock == uint32_t(kDefLitBufSize - 1);
    };
    auto flush = [&]() {
      B->symEnd[nBlocks] = k;
      B->posEnd[nBlocks] = strstart;
      nBlocks++;
      inBlock = 0;
    };
    while (strstart < n) {
      const uint32_t c = strstart / uint32_t(kDecChunk);
      if (c != curChunk) {
        // chunks [c, c + kDecRing) must be in flight or landed; chunks skipped by a long match are committed empty.
        // After a skip the ring slots about to be refilled may still be the target of copies in flight (two cp.async
        // to one address are not ordered): drain first.
        if (c != curChunk + 1u) asm volatile("cp.async.wait_group 0;" ::: "memory");
        while (fetched < c + uint32_t(kDecRing)) {
          if (fetched >= c && fetched < nChunks) {
            const uint32_t slot = fetched % uint32_t(kDecRing);
            const char* tsrc = reinterpret_cast<const char*>(table + size_t(fetched) * kDecChunk);
            const uint32_t tdst = tabBase + slot * uint32_t(kDecChunk * 4);
#pragma unroll
            for (int q = 0; q < kDecChunk * 4 / 16; q++)
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(tdst + q * 16), "l"(tsrc + q * 16) : "memory");
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(byteBase + slot * uint32_t(kDecChunk)),
                         "l"(in + size_t(fetched) * kDecChunk) : "memory");
          }
          asm volatile("cp.async.commit_group;" ::: "memory");
          fetched++;
        }
        asm volatile("cp.async.wait_group %0;" ::"n"(kDecRing - 1) : "memory");
        curChunk = c;
      }
      const uint32_t ri = strstart % uint32_t(kDecRow);
      const uint32_t curByte = byteS[lane][ri];
      const uint32_t lookahead = n - strstart;
      prevLength = matchLength;
      prevMatch = matchStart;
      matchLength = kDefMinMatch - 1;
      if (lookahead >= uint32_t(kDefMinMatch) && prevLength < L.maxLazy) {
        uint32_t w = tabS[lane][ri];
        if (w >> 31) w = prevLength >= L.goodLength ? tableQ[strstart] : (w & 0x7fffffffu);  // rare: the quarter chain differs
        const int len = int(w & 0x1ffu);
        if (len > prevLength) {
          matchLength = len;
          matchStart = strstart - (w >> 9);
          if (matchLength == kDefMinMatch && strstart - matchStart > uint32_t(kDefTooFar)) matchLength = kDefMinMatch - 1;
        }
      }
      if (prevLength >= kDefMinMatch && matchLength <= prevLength) {
        const bool bflush = tally(strstart - 1 - prevMatch, uint32_t(prevLength - kDefMinMatch));
        strstart += uint32_t(prevLength - 1);
        matchAvailable = false;
        matchLength = kDefMinMatch - 1;
        if (bflush) flush();
      } else if (matchAvailable) {
        const bool bflush = tally(0, lastByte);
        if (bflush) flush();
        strstart++;
        lastByte = curByte;
      } else {
        matchAvailable = true;
        strstart++;
        lastByte = curByte;
      }
    }
    if (matchAvailable) tally(0, lastByte);
    for (uint32_t i = k & ~7u; i < k; i++) symDist[i] = distS[lane][i & 7u];
    for (uint32_t i = k & ~15u; i < k; i++) symLc[i] = lcS[lane][i & 15u];
    flush();
    B->nBlocks = nBlocks;
    asm volatile("cp.async.wait_group 0;" ::: "memory");  // nothing of this stream may land in the next one's ring
  }
}

// emit: one CTA per stream.  The blocks of a stream are independent until their bits are laid end to end, and what a
// block costs is trees.c on ONE thread (build_tree's heap is a chain of dependent shared-memory accesses: 60 % of the
// kernel's samples sat at the barrier behind it).  So up to kEmitPar blocks are planned at once: their symbol
// histograms by all threads, then one thread per block runs def_plan_block and renders the block header (type bits +
// the three trees) into a private buffer; after that the blocks are emitted in order -- header words copied in
// parallel, symbols in parallel (every thread sizes four consecutive symbols, a block scan gives the bit offsets, the
// codes are OR-ed into the shared-memory bit window of g4_bitpack.cuh).  Adler-32 by a block reduction
// (s2 = n + sum (n-i) b_i).
namespace {
constexpr int kEmitPar = 3;  // 43 KB of M32 bytes are at most three blocks of 16,383 symbols
constexpr int kEmitHdrWords = 152;  // 3 + 14 + 19 * 3 + 316 * 14 bits at most
struct DeflateEmitShared {
  DeflateTrees T[kEmitPar];
  BitWindow W;
  uint32_t lhist[kDefLCodes + 2], dhist[kDefDCodes + 2];
  uint32_t scan[kWarps + 1];
  DeflateBlockPlan plan[kEmitPar];
  uint32_t hdr[kEmitPar][kEmitHdrWords];
  uint32_t hdrBits[kEmitPar];
  unsigned long long red[kWarps][2];
  int j;
};
struct BufOut {  // serial writer into a zeroed word buffer (the Out of def_send_all_trees)
  uint32_t* w;
  uint32_t pos;
  __device__ __forceinline__ void send_bits(uint32_t v, int n) {
    if (!n) return;
    const uint32_t i = pos >> 5, o = pos & 31;
    w[i] |= v << o;
    if (o + uint32_t(n) > 32u) w[i + 1] |= v >> (32 - o);
    pos += uint32_t(n);
  }
};
__device__ __forceinline__ uint32_t emit_sym_bits(const DeflateTrees& T, bool useStatic, uint32_t dist, uint32_t lc) {
  if (dist == 0) return useStatic ? uint32_t(def_static_llen(int(lc))) : T.ltree[lc].dl;
  const int lcode = def_length_code(int(lc));
  const int dcode = def_dist_code(int(dist - 1));
  const uint32_t l = useStatic ? uint32_t(def_static_llen(lcode + 257)) : T.ltree[lcode + 257].dl;
  const uint32_t d = useStatic ? 5u : T.dtree[dcode].dl;
  return l + uint32_t(def_length_extra(lcode)) + d + uint32_t(def_dist_extra(dcode));
}
__device__ __forceinline__ void emit_sym_put(ThreadBits& tb, const DeflateTrees& T, bool useStatic, uint32_t dist, uint32_t lc) {
  if (dist == 0) {
    if (useStatic) tb.put(def_static_lcode(int(lc)), def_static_llen(int(lc)));
    else tb.put(T.ltree[lc].fc, T.ltree[lc].dl);
    return;
  }
  const int lcode = def_length_code(int(lc));
  if (useStatic) tb.put(def_static_lcode(lcode + 257), def_static_llen(lcode + 257));
  else tb.put(T.ltree[lcode + 257].fc, T.ltree[lcode + 257].dl);
  const int lx = def_length_extra(lcode);
  if (lx) tb.put(uint32_t(int(lc) - def_length_base(lcode)), lx);
  const int d1 = int(dist - 1);
  const int dcode = def_dist_code(d1);
  if (useStatic) tb.put(def_bi_reverse(uint32_t(dcode), 5), 5);
  else tb.put(T.dtree[dcode].fc, T.dtree[dcode].dl);
  const int dx = def_dist_extra(dcode);
  if (dx) tb.put(uint32_t(d1 - def_dist_base(dcode)), dx);
}
}  // namespace

__global__ void __launch_bounds__(kThreads) deflate_emit_kernel(StagedArgs a) {
  extern __shared__ __align__(16) unsigned char emitSm[];
  DeflateEmitShared& S = *reinterpret_cast<DeflateEmitShared*>(emitSm);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const DeflateLevel L = deflate_level(a.level);
  for (;;) {
    __syncthreads();
    if (tid == 0) S.j = a.jBegin + atomicAdd(a.counters + 3, 1);
    __syncthreads();
    const int j = S.j;
    if (j >= a.jEnd) break;
    const uint32_t n = a.inLen[j];
    if (n > kDefStagedMax) continue;
    if (n == 0) { if (tid == 0) a.outLen[j] = 0; continue; }
    const uint64_t off = a.inOff[j];
    const uint8_t* in = a.inBuf + off;
    const uint16_t* symDist = a.lazy ? reinterpret_cast<const uint16_t*>(a.table + (off - a.baseOff)) : a.sorted + (off - a.baseOff);
    const uint8_t* symLc = a.lazy ? reinterpret_cast<const uint8_t*>(a.tableQ + (off - a.baseOff))
                                  : reinterpret_cast<const uint8_t*>(a.rank + (off - a.baseOff));
    const DeflateBlocks& B = a.blocks[j - a.jBegin];
    const uint32_t cap = n + uint32_t(a.capExtra);
    BitOut o;
    bitwin_reset(S.W, o, reinterpret_cast<uint32_t*>(a.outBuf + off + 112ull * uint64_t(j)), (cap + 3) >> 2);
    if (tid == 0) {
      WinSink hs{S.W.win, 0};
      hs.put(L.zlibHeader >> 8, 8);
      hs.put(L.zlibHeader & 0xffu, 8);
    }
    o.bitPos = 16;
    const uint32_t nBlocks = B.nBlocks;
    for (uint32_t b0 = 0; b0 < nBlocks; b0 += kEmitPar) {
      const uint32_t nb = nBlocks - b0 < uint32_t(kEmitPar) ? nBlocks - b0 : uint32_t(kEmitPar);
      // histograms of the batch's blocks, one after the other, into the blocks' own trees
      for (uint32_t i = 0; i < nb; i++) {
        const uint32_t sym0 = b0 + i ? B.symEnd[b0 + i - 1] : 0u, sym1 = B.symEnd[b0 + i];
        __syncthreads();
        for (int q = tid; q < kDefLCodes + 2; q += kThreads) S.lhist[q] = 0;
        if (tid < kDefDCodes + 2) S.dhist[tid] = 0;
        for (int q = tid; q < kEmitHdrWords; q += kThreads) S.hdr[i][q] = 0;
        __syncthreads();
        for (uint32_t q = sym0 + tid; q < sym1; q += kThreads) {
          const uint32_t dist = symDist[q], lc = symLc[q];
          if (dist == 0) atomicAdd(&S.lhist[lc], 1u);
          else {
            atomicAdd(&S.lhist[def_length_code(int(lc)) + 257], 1u);
            atomicAdd(&S.dhist[def_dist_code(int(dist - 1))], 1u);
          }
        }
        __syncthreads();
        for (int q = tid; q < kDefLCodes; q += kThreads) S.T[i].ltree[q].fc = uint16_t(q == 256 ? 1u : S.lhist[q]);
        if (tid < kDefDCodes) S.T[i].dtree[tid].fc = uint16_t(S.dhist[tid]);
        if (tid < kDefBlCodes) S.T[i].bltree[tid].fc = 0;
      }
      __syncthreads();
      if (lane == 0 && uint32_t(warp) < nb) {  // trees.c for block b0 + warp, and its header
        const uint32_t b = b0 + uint32_t(warp);
        DeflateState st;
        st.W = nullptr;
        st.T = &S.T[warp];
        st.optLen = st.staticLen = 0;
        const DeflateBlockPlan P = def_plan_block(st, B.posEnd[b] - (b ? B.posEnd[b - 1] : 0u), true);
        S.plan[warp] = P;
        BufOut bo{S.hdr[warp], 0};
        bo.send_bits((uint32_t(P.type) << 1) + (b + 1 == nBlocks ? 1u : 0u), 3);
        if (P.type == 2) def_send_all_trees(st, bo, P);
        S.hdrBits[warp] = bo.pos;
      }
      __syncthreads();
      for (uint32_t i = 0; i < nb; i++) {
        const uint32_t b = b0 + i;
        const uint32_t sym0 = b ? B.symEnd[b - 1] : 0u, sym1 = B.symEnd[b];
        const uint32_t pos0 = b ? B.posEnd[b - 1] : 0u, pos1 = B.posEnd[b];
        const DeflateTrees& T = S.T[i];
        bitwin_reserve(S.W, o, 8192);  // room for the block header; contains the barrier
        {
          const uint32_t hb = S.hdrBits[i];
          if (uint32_t(tid) * 32u < hb) {
            const uint32_t left = hb - uint32_t(tid) * 32u;
            ThreadBits tb;
            tb.begin(S.W, o, o.bitPos + uint32_t(tid) * 32u);
            tb.put(S.hdr[i][tid], left < 32u ? int(left) : 32);
            tb.end();
          }
          o.bitPos += hb;
        }
        __syncthreads();
        const int type = S.plan[i].type;
        if (type == 0) {
          // stored: pad to a byte boundary, LEN, NLEN, then the raw bytes (eight per thread and step)
          const uint32_t len = pos1 - pos0;
          o.bitPos = (o.bitPos + 7u) & ~7u;
          bitwin_reserve(S.W, o, 64);
          if (tid == 0) {
            WinSink hs{S.W.win, o.bitPos - o.gbase * 32u};
            hs.put(len & 0xffffu, 16);
            hs.put((~len) & 0xffffu, 16);
          }
          o.bitPos += 32;
          __syncthreads();
          for (uint32_t i0 = 0; i0 < len; i0 += kThreads * 8) {
            const uint32_t rem = len - i0;
            const uint32_t chunk = rem < uint32_t(kThreads * 8) ? rem : uint32_t(kThreads * 8);
            bitwin_reserve(S.W, o, chunk * 8);
            const uint32_t mine = i0 + uint32_t(tid) * 8u;
            if (mine < i0 + chunk) {
              ThreadBits tb;
              tb.begin(S.W, o, o.bitPos + uint32_t(tid) * 64u);
              const uint32_t cnt = (i0 + chunk - mine) < 8u ? (i0 + chunk - mine) : 8u;
              for (uint32_t q = 0; q < cnt; q++) tb.put(in[pos0 + mine + q], 8);
              tb.end();
            }
            o.bitPos += chunk * 8;
            __syncthreads();
          }
        } else {
          const bool useStatic = type == 1;
          constexpr int kIpt = 4;
          for (uint32_t k0 = sym0; k0 < sym1; k0 += kThreads * kIpt) {
            uint32_t dist[kIpt], lc[kIpt];
            uint32_t myBits = 0;
            int nv = 0;
#pragma unroll
            for (int q = 0; q < kIpt; q++) {
              const uint32_t k = k0 + uint32_t(tid) * kIpt + q;
              if (k < sym1) {
                dist[q] = symDist[k];
                lc[q] = symLc[k];
                myBits += emit_sym_bits(T, useStatic, dist[q], lc[q]);
                nv = q + 1;
              }
            }
            uint32_t chunkBits;
            const uint32_t ex = block_exclusive_scan(myBits, S.scan, &chunkBits);
            bitwin_reserve(S.W, o, chunkBits);  // 1024 symbols * 48 bits always fit an empty window
            ThreadBits tb;
            tb.begin(S.W, o, o.bitPos + ex);
#pragma unroll
            for (int q = 0; q < kIpt; q++)
              if (q < nv) emit_sym_put(tb, T, useStatic, dist[q], lc[q]);
            tb.end();
            o.bitPos += chunkBits;
            __syncthreads();
          }
          bitwin_reserve(S.W, o, 32);
          if (tid == 0) {
            WinSink es{S.W.win, o.bitPos - o.gbase * 32u};
            if (useStatic) es.put(def_static_lcode(256), 7);
            else es.put(T.ltree[256].fc, T.ltree[256].dl);
          }
          o.bitPos += useStatic ? 7u : uint32_t(T.ltree[256].dl);
          __syncthreads();
        }
      }
    }
    o.bitPos = (o.bitPos + 7u) & ~7u;  // bi_windup after the last block
    // Adler-32: s1 = 1 + sum b_i, s2 = n + sum (n - i) b_i  (mod 65521)
    unsigned long long sa = 0, sb = 0;
    for (uint32_t i = tid; i < n; i += kThreads) {
      const unsigned long long v = in[i];
      sa += v;
      sb += v * (n - i);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      sa += __shfl_down_sync(0xffffffffu, sa, d);
      sb += __shfl_down_sync(0xffffffffu, sb, d);
    }
    __syncthreads();
    if (lane == 0) { S.red[warp][0] = sa; S.red[warp][1] = sb; }
    bitwin_reserve(S.W, o, 64);
    __syncthreads();
    if (tid == 0) {
      unsigned long long ta = 1, tb2 = n;
      for (int w = 0; w < kWarps; w++) { ta += S.red[w][0]; tb2 += S.red[w][1]; }
      const uint32_t s1 = uint32_t(ta % 65521ull), s2 = uint32_t(tb2 % 65521ull);
      WinSink ts{S.W.win, o.bitPos - o.gbase * 32u};
      ts.put(s2 >> 8, 8);
      ts.put(s2 & 0xffu, 8);
      ts.put(s1 >> 8, 8);
      ts.put(s1 & 0xffu, 8);
    }
    o.bitPos += 32;
    __syncthreads();
    bitwin_finish(S.W, o);
    const uint32_t total = o.bitPos >> 3;
    if (tid == 0) a.outLen[j] = total > cap ? cap : total;
  }
}

// ---- CodecDeflate ---------------------------------------------------------------------------------------------
namespace {
struct PredResidualGet {
  TileView t;
  int pred;
  __device__ __forceinline__ int32_t operator()(uint32_t k) const {
    int r, c;
    stream_to_cell(pred, int(k), t.R, t.C, &r, &c);
    return residual_at(pred, t, r, c);
  }
};
struct NullsResidualGet {  // PredictorModelDifferencingWithNulls: one residual per cell, row-major
  TileView t;
  int32_t seed;
  __device__ __forceinline__ int32_t operator()(uint32_t k) const {
    int r = int(k) / t.C, c = int(k) - r * t.C;
    return residual_nulls_at(t, r, c, seed);
  }
};
}  // namespace

__global__ void __launch_bounds__(kThreads) deflate_m32_size_kernel(EncodeArgs a, uint32_t* inLen) {
  __shared__ uint32_t scan[kWarps + 1];
  const int tid = threadIdx.x;
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (int tIdx = blockIdx.x; tIdx < nTiles; tIdx += gridDim.x) {
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int n = t.R * t.C;
    bool sawNull = false, sawValid = false;
    for (int i = tid; i < n; i += kThreads) {
      int r = i / t.C, c = i - r * t.C;
      if (t.at(r, c) == kNull) sawNull = true; else sawValid = true;
    }
    const bool anyNull = __syncthreads_or(sawNull) != 0;
    const bool anyValid = __syncthreads_or(sawValid) != 0;
    if (!anyValid) {  // all-null tile -> null (:167-169)
      if (tid == 0) {
        a.lens[tIdx] = 0; a.preds[tIdx] = 0; a.status[tIdx] = G4_DECLINED;
        inLen[3 * tIdx] = inLen[3 * tIdx + 1] = inLen[3 * tIdx + 2] = 0;
      }
      continue;
    }
    if (anyNull) {  // only PredictorModelDifferencingWithNulls applies (:178-186): one stream, a.preds marks the case
      int nStart;
      const int32_t seed = nulls_seed(t, &nStart);
      uint32_t sz = m32_stream_size(NullsResidualGet{t, seed}, uint32_t(n), scan);
      if (tid == 0) {
        inLen[3 * tIdx] = sz; inLen[3 * tIdx + 1] = inLen[3 * tIdx + 2] = 0;
        a.preds[tIdx] = G4_PRED_DIFF_NULLS; a.status[tIdx] = G4_OK;
      }
      continue;
    }
    if (tid == 0) a.preds[tIdx] = 0;
    for (int p = 0; p < 3; p++) {
      PredResidualGet get{t, p + 1};
      uint32_t sz = m32_stream_size(get, uint32_t(n - 1), scan);
      if (tid == 0) inLen[3 * tIdx + p] = sz;
    }
    if (tid == 0) a.status[tIdx] = G4_OK;
  }
}

__global__ void __launch_bounds__(kThreads) deflate_m32_write_kernel(EncodeArgs a, const uint32_t* inLen, const uint64_t* inOff,
                                                                     uint8_t* inBuf) {
  __shared__ uint32_t scan[kWarps + 1];
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (int tIdx = blockIdx.x; tIdx < nTiles; tIdx += gridDim.x) {
    if (inLen[3 * tIdx] == 0) continue;
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int n = t.R * t.C;
    if (a.preds[tIdx] == G4_PRED_DIFF_NULLS) {
      int nStart;
      const int32_t seed = nulls_seed(t, &nStart);
      uint8_t* dst = inBuf + inOff[3 * tIdx];
      uint32_t w = m32_stream_write(NullsResidualGet{t, seed}, uint32_t(n), dst, scan);
      if (threadIdx.x < 16) dst[w + threadIdx.x] = 0;
      continue;
    }
    for (int p = 0; p < 3; p++) {
      PredResidualGet get{t, p + 1};
      uint8_t* dst = inBuf + inOff[3 * tIdx + p];
      uint32_t w = m32_stream_write(get, uint32_t(n - 1), dst, scan);
      if (threadIdx.x < 16) dst[w + threadIdx.x] = 0;  // the pre-filter of longest_match may look 2 bytes past the end
    }
  }
}

__global__ void __launch_bounds__(kThreads) deflate_pick_kernel(EncodeArgs a, const uint32_t* inLen, const uint64_t* inOff,
                                                                const uint8_t* outBuf, const uint32_t* outLen) {
  const int tid = threadIdx.x;
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (int tIdx = blockIdx.x; tIdx < nTiles; tIdx += gridDim.x) {
    if (inLen[3 * tIdx] == 0) continue;
    // CodecDeflate.encode: Differencing, Linear, Triangle; keep the strictly smallest packing (:176-199)
    uint32_t best = 0xffffffffu;
    int win = -1;
    for (int p = 0; p < 3; p++) {
      uint32_t dN = outLen[3 * tIdx + p];
      if (dN > 0 && dN < best) { best = dN; win = p; }  // dN <= 0: "deflate failed" -> candidate skipped (:211-214)
    }
    if (win < 0) {
      if (tid == 0) { a.lens[tIdx] = 0; a.preds[tIdx] = 0; a.status[tIdx] = G4_DECLINED; }
      continue;
    }
    const int j = 3 * tIdx + win;
    const uint32_t len = best + 10u;
    const bool fits = len <= a.slotBytes;
    const bool nulls = a.preds[tIdx] == G4_PRED_DIFF_NULLS;
    const TileView t = tile_view(a.band, a.grid, tIdx);
    int nStart = 0;
    const int32_t seedNulls = nulls ? nulls_seed(t, &nStart) : 0;
    const int predCode = nulls ? G4_PRED_DIFF_NULLS : win + 1;
    if (fits) {
      uint8_t* slot = a.slots + size_t(tIdx) * a.slotBytes;
      const uint8_t* src = outBuf + inOff[j] + 112ull * uint64_t(j);
      if (tid == 0) {
        const uint32_t seed = nulls ? uint32_t(seedNulls) : uint32_t(t.at(0, 0)), nM32 = inLen[j];
        slot[0] = uint8_t(a.codecIndex);
        slot[1] = uint8_t(predCode);
        for (int k = 0; k < 4; k++) { slot[2 + k] = uint8_t(seed >> (8 * k)); slot[6 + k] = uint8_t(nM32 >> (8 * k)); }
      }
      for (uint32_t i = tid; i < best; i += kThreads) slot[10 + i] = src[i];
    }
    __syncthreads();
    if (tid == 0) { a.lens[tIdx] = len; a.preds[tIdx] = uint8_t(predCode); a.status[tIdx] = fits ? G4_OK : G4_ERR_CAPACITY; }
  }
}

// ---- CodecFloat -------------------------------------------------------------------------------------------------
// Streams of tile t: 5t+0 sign bitmap ((n+7)/8 bytes, cell i -> bit i LSB-first), 5t+1 exponent bytes, 5t+2..4 the
// mantissa bytes (high 7 bits, middle, low) as row-wise byte differences; the first byte of a row differences
// against the first byte of the previous row (row 0 against 0).
__global__ void float_plane_size_kernel(int nTiles, uint32_t n, uint32_t* inLen) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= 5 * nTiles) return;
  inLen[j] = (j % 5 == 0) ? (n + 7u) / 8u : n;
}

__global__ void __launch_bounds__(kThreads) float_plane_write_kernel(EncodeArgs a, const uint64_t* inOff, uint8_t* inBuf) {
  const int tid = threadIdx.x;
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (int tIdx = blockIdx.x; tIdx < nTiles; tIdx += gridDim.x) {
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int R = t.R, C = t.C, n = R * C;
    uint8_t* pl[5];
    for (int p = 0; p < 5; p++) pl[p] = inBuf + inOff[5 * tIdx + p];
    const int nSignBytes = (n + 7) / 8;
    for (int b = tid; b < nSignBytes; b += kThreads) {
      uint32_t v = 0;
      for (int i = 0; i < 8; i++) {
        int k = 8 * b + i;
        if (k < n) { int r = k / C, c = k - r * C; v |= (uint32_t(t.at(r, c)) >> 31) << i; }
      }
      pl[0][b] = uint8_t(v);
    }
    for (int k = tid; k < n; k += kThreads) {
      int r = k / C, c = k - r * C;
      uint32_t bits = uint32_t(t.at(r, c));
      uint32_t prior = c > 0 ? uint32_t(t.at(r, c - 1)) : r > 0 ? uint32_t(t.at(r - 1, 0)) : 0u;
      pl[1][k] = uint8_t(bits >> 23);
      pl[2][k] = uint8_t(((bits >> 16) & 0x7fu) - ((prior >> 16) & 0x7fu));
      pl[3][k] = uint8_t((bits >> 8) - (prior >> 8));
      pl[4][k] = uint8_t(bits - prior);
    }
    if (tid < 16) {
      pl[0][nSignBytes + tid] = 0;
      for (int p = 1; p < 5; p++) pl[p][n + tid] = 0;
    }
  }
}

__global__ void __launch_bounds__(kThreads) float_pick_kernel(EncodeArgs a, const uint64_t* inOff, const uint8_t* outBuf,
                                                              const uint32_t* outLen) {
  const int tid = threadIdx.x;
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (int tIdx = blockIdx.x; tIdx < nTiles; tIdx += gridDim.x) {
    uint32_t dN[5], total = 2;
    bool failed = false;
    for (int p = 0; p < 5; p++) {
      dN[p] = outLen[5 * tIdx + p];
      if (dN[p] == 0) failed = true;  // doDeflate throws "Deflate failed"
      total += 4u + dN[p];
    }
    const bool fits = total <= a.slotBytes;
    if (!failed && fits) {
      uint8_t* slot = a.slots + size_t(tIdx) * a.slotBytes;
      if (tid == 0) { slot[0] = uint8_t(a.codecIndex); slot[1] = 0; }
      uint32_t off = 2;
      for (int p = 0; p < 5; p++) {
        const int j = 5 * tIdx + p;
        const uint8_t* src = outBuf + inOff[j] + 112ull * uint64_t(j);
        if (tid < 4) slot[off + tid] = uint8_t(dN[p] >> (8 * tid));
        off += 4;
        for (uint32_t i = tid; i < dN[p]; i += kThreads) slot[off + i] = src[i];
        off += dN[p];
      }
    }
    if (tid == 0) {
      a.lens[tIdx] = failed ? 0u : total;
      a.preds[tIdx] = 0;
      a.status[tIdx] = failed ? G4_DECLINED : fits ? G4_OK : G4_ERR_CAPACITY;
    }
  }
}

// ---- launchers ------------------------------------------------------------------------------------------------------
cudaError_t launch_stream_offsets(const uint32_t* inLen, uint64_t* inOff, int nStreams, uint64_t* total, cudaStream_t s) {
  stream_offsets_kernel<<<1, kThreads, 0, s>>>(inLen, inOff, nStreams, total);
  return cudaGetLastError();
}
cudaError_t launch_deflate_streams(const StreamArgs& a, int nWorkers, cudaStream_t s) {
  deflate_streams_kernel<<<(nWorkers + 31) / 32, 32, 0, s>>>(a);
  return cudaGetLastError();
}
uint32_t deflate_staged_max() { return kDefStagedMax; }
size_t deflate_blocks_bytes() { return sizeof(DeflateBlocks); }
cudaError_t launch_deflate_staged(const StagedArgs& a, int smCount, cudaStream_t s) {
  static std::atomic<uint64_t> attr{0};
  cudaError_t ea = once_per_device(attr, [] {
    return cudaFuncSetAttribute(deflate_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDefWSize * 2);
  });
  if (ea != cudaSuccess) return ea;
  const int nChunk = a.jEnd - a.jBegin;
  const int sortCtas = nChunk < smCount * 3 ? nChunk : smCount * 3;
  deflate_sort_kernel<<<sortCtas, kSortThreads, kDefWSize * 2, s>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (a.lazy) {
    const int warps = nChunk < smCount * 48 ? nChunk : smCount * 48;
    deflate_lazy_kernel<<<(warps + 3) / 4, 128, 0, s>>>(a);
  } else {
    // match: shared memory = the candidate window + the stream's table (4 bytes per position) when that fits
    size_t win = size_t(128 + 1920) * 16;                // two groups of (128 + 896) slots: the same
    const size_t winBig = size_t(2) * (128 + 1408) * 16;  // two groups of 1,536 slots
    const size_t smMax = 227 * 1024 - 2048;
    size_t tabBytes = (size_t(a.maxLen) * 4 + 15) & ~size_t(15);
    if (win + tabBytes > smMax) tabBytes = 0;  // too long: scattered stores
    int perSm = int(smMax / (win + tabBytes));
    if (perSm > 8) perSm = 8;
    // one CTA per SM anyway: the larger windows if they fit beside the table (fewer rounds, less of each window re-filled)
    const bool big = perSm == 1 && winBig + tabBytes <= smMax;
    if (big) win = winBig;
    const size_t sm = win + tabBytes;
    const int threads = perSm == 1 ? 1024 : perSm <= 3 ? 512 : 256;
    const int ctas = nChunk < smCount * perSm ? nChunk : smCount * perSm;
    static std::atomic<uint64_t> attrW{0};
    ea = once_per_device(attrW, [] {
      const int cap = 227 * 1024 - 2048;
      cudaError_t e1 = cudaFuncSetAttribute(deflate_match_window_kernel<1920, 1, 512, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
      if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(deflate_match_window_kernel<1408, 2, 1024, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
      if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(deflate_match_window_kernel<896, 2, 1024, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap);
      return e1;
    });
    if (ea != cudaSuccess) return ea;
    const uint32_t cap32 = uint32_t(tabBytes / 4);
    if (big) deflate_match_window_kernel<1408, 2, 1024, 1><<<ctas, threads, sm, s>>>(a, cap32);
    else if (threads == 1024) deflate_match_window_kernel<896, 2, 1024, 1><<<ctas, threads, sm, s>>>(a, cap32);
    else deflate_match_window_kernel<1920, 1, 512, 3><<<ctas, threads, sm, s>>>(a, cap32);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    deflate_decide_ring_kernel<<<(nChunk + 31) / 32, 32, 0, s>>>(a);
  }
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  static std::atomic<uint64_t> attrE{0};
  ea = once_per_device(attrE, [] {
    return cudaFuncSetAttribute(deflate_emit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(DeflateEmitShared)));
  });
  if (ea != cudaSuccess) return ea;
  deflate_emit_kernel<<<nChunk < smCount * 8 ? nChunk : smCount * 8, kThreads, sizeof(DeflateEmitShared), s>>>(a);
  return cudaGetLastError();
}
cudaError_t launch_deflate_m32_size(const EncodeArgs& a, uint32_t* inLen, int nCtas, cudaStream_t s) {
  deflate_m32_size_kernel<<<nCtas, kThreads, 0, s>>>(a, inLen);
  return cudaGetLastError();
}
cudaError_t launch_deflate_m32_write(const EncodeArgs& a, const uint32_t* inLen, const uint64_t* inOff, uint8_t* inBuf, int nCtas,
                                     cudaStream_t s) {
  deflate_m32_write_kernel<<<nCtas, kThreads, 0, s>>>(a, inLen, inOff, inBuf);
  return cudaGetLastError();
}
cudaError_t launch_deflate_pick(const EncodeArgs& a, const uint32_t* inLen, const uint64_t* inOff, const uint8_t* outBuf,
                                const uint32_t* outLen, int nCtas, cudaStream_t s) {
  deflate_pick_kernel<<<nCtas, kThreads, 0, s>>>(a, inLen, inOff, outBuf, outLen);
  return cudaGetLastError();
}
cudaError_t launch_float_plane_size(int nTiles, uint32_t n, uint32_t* inLen, cudaStream_t s) {
  float_plane_size_kernel<<<(5 * nTiles + 255) / 256, 256, 0, s>>>(nTiles, n, inLen);
  return cudaGetLastError();
}
cudaError_t launch_float_plane_write(const EncodeArgs& a, const uint64_t* inOff, uint8_t* inBuf, int nCtas, cudaStream_t s) {
  float_plane_write_kernel<<<nCtas, kThreads, 0, s>>>(a, inOff, inBuf);
  return cudaGetLastError();
}
cudaError_t launch_float_pick(const EncodeArgs& a, const uint64_t* inOff, const uint8_t* outBuf, const uint32_t* outLen, int nCtas,
                              cudaStream_t s) {
  float_pick_kernel<<<nCtas, kThreads, 0, s>>>(a, inOff, outBuf, outLen);
  return cudaGetLastError();
}

}  // namespace g4
