// g4_huffman.cu -- CodecHuffman (legacy byte-alphabet Huffman over M32 predictor residuals) on sm_100a.
//
// Reference: compress/CodecHuffman.java:70-153, compress/HuffmanEncoder.java:124-305,
//            compress/HuffmanDecoder.java:65-187   (under /root/reference/core/src/main/java/org/gridfour/).
//
// Encode, one persistent CTA per tile at a time:
//   pass 1  coalesced sweep of the tile: residuals of all three predictors per cell, M32 lengths/bytes,
//           three 256-bin shared-memory histograms
//   trees   rank sort of (count,symbol); size of every candidate = header + tree + sum of branch counts;
//           the winner's tree is rebuilt by one thread with the reference's tie-breaking (a new branch
//           goes in front of every node of equal count)
//   pass 2  the winner's residuals in stream order -> M32 bytes -> codes; bit offsets from a block scan;
//           bits are OR-ed into a shared-memory window and flushed with coalesced word stores
// Decode:
//   tree parse by one thread -> 11-bit lookup table filled by all threads; text decoded by all threads as
//   self-synchronising sub-sequences (speculative start, iterate until hand-over positions agree), count
//   scan -> byte offsets -> second pass writes the M32 bytes; then g4_predict.cuh.
#include "g4_kernels.h"
#include "g4_predict.cuh"
#include "g4_huffdec.cuh"
#include "g4_huff_fast.cuh"
#include "g4_huff2.cuh"

namespace g4 {

// =================================================================================================
// Encode
// =================================================================================================
namespace {

constexpr int kWinWords = 4096;                 // 16 KB output window
constexpr uint32_t kWinBits = kWinWords * 32u;
constexpr int kEmitItems = 8;                   // residuals per thread per chunk

struct HuffEncShared {
  uint32_t hist[3][256];
  uint32_t skey[3][256];     // sorted (count<<8 | symbol), ascending
  uint32_t bq[3][256];       // branch-count queues for the size-only merges
  uint32_t bcount[256];      // winner: branch counts by creation order
  uint16_t bqueue[256];      // winner: branch ids in list order
  uint16_t left[256], right[256];
  uint64_t code[512];        // node code, path order LSB first (leaves 0..255 by symbol, branches 256+id)
  uint8_t len[512];
  uint32_t win[kWinWords + 4];
  uint32_t scan[kWarps + 1];
  uint32_t nLeaf[3];
  unsigned long long textBits[3];
  uint32_t nBytes[3];
  int hasNull;
  int winner;
};

// size-only Huffman merge: returns the sum of all branch counts (== text bits).  Tie order is irrelevant
// for the total.  keys ascending, first `256-L` entries have count 0.
__device__ unsigned long long merge_size_only(const uint32_t* skey, uint32_t* bq, int L) {
  int li = 256 - L, bi = 0, bt = 0;
  unsigned long long total = 0;
  for (int m = 0; m < L - 1; m++) {
    uint32_t c[2];
#pragma unroll
    for (int k = 0; k < 2; k++) {
      bool takeBranch = (bi < bt) && (li > 255 || bq[bi] <= (skey[li] >> 8));
      if (takeBranch) c[k] = bq[bi++];
      else c[k] = skey[li++] >> 8;
    }
    uint32_t s = c[0] + c[1];
    bq[bt++] = s;
    total += s;
  }
  return total;
}

// Winner tree with the reference's list-insertion rule (HuffmanEncoder.java:165-194): a new branch is
// placed in front of the first remaining node whose count is >= its own, so among equal counts the order
// is: newest branch ... oldest branch, then leaves by symbol.
__device__ void build_winner_tree(HuffEncShared& S, int p, int L) {
  const uint32_t* skey = S.skey[p];
  int li = 256 - L, bi = 0, bt = 0, nb = 0;
  for (int m = 0; m < L - 1; m++) {
    uint16_t node[2];
    uint32_t cnt[2];
#pragma unroll
    for (int k = 0; k < 2; k++) {
      bool takeBranch = (bi < bt) && (li > 255 || S.bcount[S.bqueue[bi]] <= (skey[li] >> 8));
      if (takeBranch) { uint16_t id = S.bqueue[bi++]; node[k] = 256 + id; cnt[k] = S.bcount[id]; }
      else { uint32_t key = skey[li++]; node[k] = key & 0xff; cnt[k] = key >> 8; }
    }
    int id = nb++;
    uint32_t s = cnt[0] + cnt[1];
    S.bcount[id] = s;
    S.left[id] = node[0];
    S.right[id] = node[1];
    int pos = bt;
    while (pos > bi && S.bcount[S.bqueue[pos - 1]] >= s) { S.bqueue[pos] = S.bqueue[pos - 1]; pos--; }
    S.bqueue[pos] = uint16_t(id);
    bt++;
  }
  // depths and codes, root first (children are always created before their parent)
  int root = 256 + (L - 2);
  S.len[root] = 0;
  S.code[root] = 0;
  for (int id = L - 2; id >= 0; id--) {
    int n = 256 + id;
    uint8_t l = S.len[n];
    uint64_t c = S.code[n];
    S.len[S.left[id]] = l + 1;
    S.code[S.left[id]] = c;
    S.len[S.right[id]] = l + 1;
    S.code[S.right[id]] = c | (uint64_t(1) << l);
  }
}

// header (CodecHuffman.java:121-130) + pre-order tree (HuffmanEncoder.java:221-294) into the window
__device__ uint32_t write_header_and_tree(HuffEncShared& S, int codecIndex, int pred, int32_t seed, uint32_t nM32, int L,
                                          int singleSymbol) {
  BitSink sink{S.win, 0};
  sink.put(uint32_t(codecIndex) & 0xff, 8);
  sink.put(uint32_t(pred), 8);
  sink.put(uint32_t(seed), 32);
  sink.put(nM32, 32);
  if (L == 1) {  // HuffmanEncoder.java:147-157
    sink.put(0, 8);
    sink.put(1, 1);
    sink.put(uint32_t(singleSymbol), 8);
    return sink.pos;
  }
  sink.put(uint32_t(L - 1), 8);
  uint16_t stack[256];
  int sp = 0;
  stack[sp++] = uint16_t(256 + (L - 2));
  while (sp > 0) {
    uint16_t n = stack[--sp];
    if (n < 256) { sink.put(1, 1); sink.put(n, 8); }
    else { sink.put(0, 1); stack[sp++] = S.right[n - 256]; stack[sp++] = S.left[n - 256]; }
  }
  return sink.pos;
}

// Flush the complete words of the window to the tile's slot and re-base the window.
// All threads call.  bitPos = total bits produced so far; *gbase = global word index of win[0].
__device__ void window_flush(HuffEncShared& S, uint32_t* outWords, uint32_t bitPos, uint32_t* gbase, uint32_t capWords) {
  __syncthreads();
  uint32_t nWords = (bitPos >> 5) - *gbase;
  for (uint32_t i = threadIdx.x; i < nWords; i += kThreads)
    if (*gbase + i < capWords) outWords[*gbase + i] = S.win[i];
  uint32_t carry = S.win[nWords];
  __syncthreads();
  for (uint32_t i = threadIdx.x; i < kWinWords + 4; i += kThreads) S.win[i] = 0;
  __syncthreads();
  if (threadIdx.x == 0) S.win[0] = carry;
  *gbase += nWords;
  __syncthreads();
}

// Emit `count` residuals starting at stream index k0 (IPT consecutive per thread).  Returns false (for
// IPT > 1 only) when the chunk cannot fit the window even after a flush; nothing is written then.
template <int IPT>
__device__ bool emit_chunk(HuffEncShared& S, const TileView& t, int pred, int32_t seed, uint32_t k0, uint32_t count, uint32_t* outWords,
                           uint32_t capWords, uint32_t* bitPos, uint32_t* gbase) {
  uint64_t packed[IPT];
  int nb[IPT];
  uint32_t myBits = 0;
  const uint32_t kBase = k0 + threadIdx.x * IPT;
#pragma unroll
  for (int j = 0; j < IPT; j++) {
    nb[j] = 0;
    packed[j] = 0;
    uint32_t k = kBase + j;
    if (k < k0 + count) {
      int r, c;
      stream_to_cell(pred, int(k), t.R, t.C, &r, &c);
      int32_t res = pred == G4_PRED_DIFF_NULLS ? residual_nulls_at(t, r, c, seed) : residual_at(pred, t, r, c);
      nb[j] = m32_encode(res, &packed[j]);
      for (int q = 0; q < nb[j]; q++) myBits += S.len[(packed[j] >> (8 * q)) & 0xff];
    }
  }
  uint32_t chunkBits;
  uint32_t ex = block_exclusive_scan(myBits, S.scan, &chunkBits);
  if (((*bitPos + chunkBits + 31) >> 5) + 1 - *gbase > uint32_t(kWinWords)) {
    window_flush(S, outWords, *bitPos, gbase, capWords);
    if (((*bitPos + chunkBits + 31) >> 5) + 1 - *gbase > uint32_t(kWinWords)) return false;
  }
  uint32_t pos = *bitPos + ex;
  uint32_t w = (pos >> 5) - *gbase;
  int nacc = int(pos & 31);
  uint64_t acc = 0;
  bool first = true;
#pragma unroll
  for (int j = 0; j < IPT; j++) {
    for (int q = 0; q < nb[j]; q++) {
      uint32_t sym = uint32_t(packed[j] >> (8 * q)) & 0xff;
      uint64_t c = S.code[sym];
      int l = S.len[sym];
      while (l > 0) {
        int take = l < 64 - nacc ? l : 64 - nacc;
        uint64_t part = take == 64 ? c : (c & ((uint64_t(1) << take) - 1));
        acc |= part << nacc;
        nacc += take;
        l -= take;
        c = take == 64 ? 0 : (c >> take);
        while (nacc >= 32) {
          if (first) { atomicOr(&S.win[w], uint32_t(acc)); first = false; }
          else S.win[w] = uint32_t(acc);
          w++;
          acc >>= 32;
          nacc -= 32;
        }
      }
    }
  }
  if (nacc > 0 && acc != 0) atomicOr(&S.win[w], uint32_t(acc));
  *bitPos += chunkBits;
  return true;
}

}  // namespace

__global__ void __launch_bounds__(kThreads) huffman_encode_kernel(EncodeArgs a) {
  extern __shared__ __align__(16) unsigned char smemRaw[];
  HuffEncShared& S = *reinterpret_cast<HuffEncShared*>(smemRaw);
  __shared__ int sTile;
  const int tid = threadIdx.x;
  const int nTiles = a.band.tiles_down * a.band.tiles_across;
  for (;;) {
    __syncthreads();
    if (tid == 0) sTile = atomicAdd(a.counter, 1);
    __syncthreads();
    const int tIdx = sTile;
    if (tIdx >= nTiles) break;
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int R = t.R, C = t.C, n = R * C;
    uint8_t* slot = a.slots + size_t(tIdx) * a.slotBytes;
    uint32_t* outWords = reinterpret_cast<uint32_t*>(slot);
    const uint32_t capWords = uint32_t(a.slotBytes / 4);

    for (int i = tid; i < 3 * 256; i += kThreads) (&S.hist[0][0])[i] = 0;
    for (int i = tid; i < kWinWords + 4; i += kThreads) S.win[i] = 0;
    if (tid == 0) S.hasNull = 0;
    __syncthreads();

    // ---- pass 1: histograms of the M32 bytes of all three predictors -------------------------------
    bool sawNull = false, sawValid = false;
    for (int i = tid; i < n; i += kThreads) {
      int r = i / C, c = i - r * C;
      if (t.at(r, c) == kNull) sawNull = true; else sawValid = true;
      if (i == 0) continue;
#pragma unroll
      for (int p = 0; p < 3; p++) {
        uint64_t packed;
        int nb = m32_encode(residual_at(p + 1, t, r, c), &packed);
        for (int q = 0; q < nb; q++) atomicAdd(&S.hist[p][(packed >> (8 * q)) & 0xff], 1u);
      }
    }
    if (sawNull) S.hasNull = 1;
    const bool anyValid = __syncthreads_or(sawValid ? 1 : 0) != 0;
    if (!anyValid) {  // all-null tile -> null (CodecHuffman.java:80-82)
      if (tid == 0) { a.lens[tIdx] = 0; a.status[tIdx] = G4_DECLINED; a.preds[tIdx] = 0; }
      continue;
    }
    const bool hasNull = S.hasNull != 0;
    int32_t seedNulls = 0;
    if (hasNull) {
      // only PredictorModelDifferencingWithNulls supports nulls (CodecHuffman.java:91-99): one candidate, kept in slot 0
      int nStart;
      seedNulls = nulls_seed(t, &nStart);
      for (int i = tid; i < 3 * 256; i += kThreads) (&S.hist[0][0])[i] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += kThreads) {
        int r = i / C, c = i - r * C;
        uint64_t packed;
        int nb = m32_encode(residual_nulls_at(t, r, c, seedNulls), &packed);
        for (int q = 0; q < nb; q++) atomicAdd(&S.hist[0][(packed >> (8 * q)) & 0xff], 1u);
      }
      __syncthreads();
    }

    // ---- rank sort of (count<<8|symbol) for the three histograms ------------------------------------
    {
      uint32_t key[3];
      int rank[3] = {0, 0, 0};
#pragma unroll
      for (int p = 0; p < 3; p++) key[p] = (S.hist[p][tid] << 8) | uint32_t(tid);
      for (int j = 0; j < 256; j++) {
#pragma unroll
        for (int p = 0; p < 3; p++) {
          uint32_t other = (S.hist[p][j] << 8) | uint32_t(j);
          rank[p] += other < key[p];
        }
      }
#pragma unroll
      for (int p = 0; p < 3; p++) S.skey[p][rank[p]] = key[p];
    }
    __syncthreads();
    // ---- candidate sizes ------------------------------------------------------------------------------
    if ((tid & 31) == 0 && (tid >> 5) < 3) {
      int p = tid >> 5;
      int L = 0;
      uint32_t nBytes = 0;
      for (int j = 0; j < 256; j++) { uint32_t c = S.skey[p][j] >> 8; L += c > 0; nBytes += c; }
      S.nLeaf[p] = L;
      S.nBytes[p] = nBytes;
      S.textBits[p] = L >= 2 ? merge_size_only(S.skey[p], S.bq[p], L) : 0ull;
    }
    __syncthreads();
    if (tid == 0) {
      // CodecHuffman.java:89-112: Differencing, Linear, Triangle; keep the strictly smallest byte length
      unsigned long long best = ~0ull;
      int win = 0;
      for (int p = 0; p < (hasNull ? 1 : 3); p++) {
        int L = S.nLeaf[p];
        unsigned long long bits = 80ull + (L == 1 ? 17ull : 8ull + 9ull * L + (L - 1) + S.textBits[p]);
        unsigned long long bytes = (bits + 7) / 8;
        if (bytes < best) { best = bytes; win = p; }
      }
      S.winner = win;
      int L = S.nLeaf[win];
      if (L >= 2) build_winner_tree(S, win, L);
      const int predCode = hasNull ? G4_PRED_DIFF_NULLS : win + 1;
      uint32_t hdrBits = write_header_and_tree(S, a.codecIndex, predCode, hasNull ? seedNulls : t.at(0, 0), S.nBytes[win], L,
                                               int(S.skey[win][255] & 0xff));
      S.scan[kWarps] = hdrBits;
      a.lens[tIdx] = uint32_t(best);
      a.preds[tIdx] = uint8_t(predCode);
      a.status[tIdx] = best <= a.slotBytes ? G4_OK : G4_ERR_CAPACITY;
    }
    __syncthreads();
    const int win = S.winner;
    const int L = S.nLeaf[win];
    uint32_t bitPos = S.scan[kWarps];
    uint32_t gbase = 0;
    const uint32_t nRes = hasNull ? uint32_t(n) : uint32_t(n - 1);
    const int predEmit = hasNull ? G4_PRED_DIFF_NULLS : win + 1;
    if (L >= 2) {
      // ---- pass 2: emit the winner's text --------------------------------------------------------------
      for (uint32_t k0 = 0; k0 < nRes; k0 += kThreads * kEmitItems) {
        uint32_t count = nRes - k0 < uint32_t(kThreads * kEmitItems) ? nRes - k0 : uint32_t(kThreads * kEmitItems);
        if (!emit_chunk<kEmitItems>(S, t, predEmit, seedNulls, k0, count, outWords, capWords, &bitPos, &gbase)) {
          for (uint32_t s0 = 0; s0 < count; s0 += kThreads) {
            uint32_t c1 = count - s0 < uint32_t(kThreads) ? count - s0 : uint32_t(kThreads);
            emit_chunk<1>(S, t, predEmit, seedNulls, k0 + s0, c1, outWords, capWords, &bitPos, &gbase);
          }
        }
      }
    }
    // final flush including the partial last word
    __syncthreads();
    {
      uint32_t nWords = ((bitPos + 31) >> 5) - gbase;
      for (uint32_t i = tid; i < nWords; i += kThreads)
        if (gbase + i < capWords) outWords[gbase + i] = S.win[i];
    }
  }
}

// =================================================================================================
// Decode (stream decoder in g4_huffdec.cuh)
// =================================================================================================
// stageWords: capacity of the fast decoder's staging buffer (dynamic shared memory sized by the launcher from the tile
// size); a packing that does not fit, or is not 4-byte aligned, takes the general decoder over HBM.
__global__ void __launch_bounds__(kThreads, 4) huffman_decode_kernel(DecodeArgs a, uint32_t stageWords) {
  extern __shared__ __align__(16) unsigned char huffDecSmem[];
  HuffDecShared& S = *reinterpret_cast<HuffDecShared*>(huffDecSmem);
  HuffFastShared& F = *reinterpret_cast<HuffFastShared*>(huffDecSmem);
  __shared__ uint32_t scanSm[kWarps + 1];
  __shared__ int sTile;
  const int tid = threadIdx.x;
  for (;;) {
    __syncthreads();
    if (tid == 0) sTile = atomicAdd(a.counter, 1);
    __syncthreads();
    const int li = sTile;
    if (li >= *a.listCount) break;
    const int tIdx = a.list[li];
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int n = t.R * t.C;
    const uint8_t* packing = a.arena + a.offsets[tIdx];
    const uint32_t len = a.lens[tIdx];
    int status = G4_OK;
    // CodecHuffman.decode header (CodecHuffman.java:134-143)
    int pred = len >= 10 ? int(packing[1]) : 0;
    int32_t seed = len >= 10 ? int32_t(load_le32(packing + 2)) : 0;
    uint32_t nM32 = len >= 10 ? load_le32(packing + 6) : 0;
    const uint32_t expect = pred == G4_PRED_DIFF_NULLS ? uint32_t(n) : uint32_t(n - 1);
    if (len < 12 || pred < 1 || pred > 4 || nM32 < expect || nM32 > uint32_t(6 * n)) status = G4_ERR_FORMAT;
    if (status == G4_OK) {
      uint8_t* m32 = a.scratch + size_t(blockIdx.x) * a.scratchStride;
      uint32_t endBit;
      bool ok;
      const uint32_t nW = (len - 8u + 3u) >> 2;  // words from byte 8 (4-byte aligned) to the end of the packing
      if ((reinterpret_cast<uintptr_t>(packing) & 3) == 0 && nW <= stageWords) {
        const uint32_t* g = reinterpret_cast<const uint32_t*>(packing + 8);
        for (uint32_t i = tid; i < nW; i += kThreads) F.sw[i] = __ldg(g + i);
        if (tid < 8) F.sw[nW + tid] = 0;
        __syncthreads();
        if (tid == 0 && (len & 3)) F.sw[nW - 1] &= (1u << (8 * (len & 3))) - 1u;  // bytes past the packing read as zero
        ok = huff_fast_decode_stream(F, 16u, (len - 8u) * 8u, nM32, m32, &endBit);
      } else {
        BitSrc src;
        src.init(packing + 10, len - 10);
        ok = huffman_decode_stream(S, src, 0, nM32, m32, &endBit);
      }
      if (!ok) status = G4_ERR_FORMAT;
      else {
        __syncthreads();
        if (!m32_parse_to_cells(m32, nM32, pred, t, expect, scanSm)) status = G4_ERR_FORMAT;
        else {
          __syncthreads();
          if (pred == G4_PRED_DIFF_NULLS) predictor_inverse_nulls(t, seed);
          else {
            if (tid == 0) t.at(0, 0) = seed;
            __syncthreads();
            predictor_inverse(pred, t, scanSm);
          }
        }
      }
    }
    if (tid == 0) a.status[tIdx] = status;
  }
}

// =================================================================================================
// Tree kernel of the fused fast path: ONE THREAD per tile parses the legacy Huffman tree (a serial job of a few hundred
// dependent steps) straight from the packing in global memory and leaves kid / leafSym / H2TreeMeta in a per-tile record,
// so that the decode CTAs load 3 KB instead of waiting for one of their threads.  Ten thousand parses run side by side.
__global__ void __launch_bounds__(64) huffman2_tree_kernel(DecodeArgs a, uint8_t* trees) {
  const int li = blockIdx.x * blockDim.x + threadIdx.x;
  if (li >= *a.listCount) return;
  const int tIdx = a.list[li];
  const uint8_t* packing = a.arena + a.offsets[tIdx];
  const uint32_t len = a.lens[tIdx];
  uint8_t* rec = trees + size_t(tIdx) * kH2TreeBytes;
  H2TreeMeta M;
  M.treeBits = 0;
  M.nLeaf = 0;
  M.single = -1;
  M.error = 1;
  if (len >= 12) {
    // words of the packing from its 4-byte line start; the last, partial word is assembled from bytes
    const uint32_t delta = uint32_t(reinterpret_cast<uintptr_t>(packing) & 3u);
    const uint32_t* gw = reinterpret_cast<const uint32_t*>(packing - delta);
    const uint32_t span = len + delta;
    auto word = [&](uint32_t i) -> uint32_t {
      if (4u * i + 4u <= span) return __ldg(gw + i);
      uint32_t v = 0;
      for (uint32_t b = 0; b < 4u; b++)
        if (4u * i + b < span) v |= uint32_t(packing[4u * i + b - delta]) << (8u * b);
      return v;
    };
    uint16_t pstack[64];
    h2_parse_tree(reinterpret_cast<uint16_t(*)[2]>(rec), reinterpret_cast<int16_t*>(rec + 2048), pstack, M, word, (delta + 10u) * 8u, span * 8u);
    M.treeBits -= 8u * delta;  // bit position inside the packing
  }
  *reinterpret_cast<H2TreeMeta*>(rec + 3072) = M;
}

// =================================================================================================
// Fused fast path (g4_huff2.cuh): Triangle predictor + one-byte M32 codes finished in shared memory; everything else is
// appended to defer[] for huffman_decode_kernel.  spill: kH2MaxSub * kH2SpillWords words per CTA.
template <int NT>
__global__ void __launch_bounds__(NT, NT == 512 ? 2 : 4)
    huffman2_decode_kernel(DecodeArgs a, Huff2Geom g, uint32_t* spill, const uint8_t* trees, int* defer, int* deferCount) {
  extern __shared__ __align__(128) unsigned char h2Smem[];
  Huff2Shared& S = *reinterpret_cast<Huff2Shared*>(h2Smem);
  uint32_t* sw = reinterpret_cast<uint32_t*>(h2Smem + ((sizeof(Huff2Shared) + 127) & ~size_t(127)));
  uint8_t* m32 = reinterpret_cast<uint8_t*>(sw) + g.stageBytes + 16;  // 16 bytes in front: the Triangle pass reads m32[-4 ..]
  __shared__ int sTile[2];
  __shared__ __align__(8) uint64_t sBar;
  const int tid = threadIdx.x;
  const uint32_t bar = h2_smem_u32(&sBar);
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(1));
    asm volatile("fence.mbarrier_init.release.cluster;");
    sTile[0] = atomicAdd(a.counter, 1);
  }
  __syncthreads();
  uint32_t parity = 0;
  uint32_t* spillArea = spill + size_t(blockIdx.x) * (kH2MaxSub * kH2SpillWords);
  for (int phase = 0;; phase ^= 1) {
    const int li = sTile[phase];
    if (li >= *a.listCount) break;
    if (tid == 0) sTile[phase ^ 1] = atomicAdd(a.counter, 1);  // the tile after this one, read after this iteration's barriers
    const int tIdx = a.list[li];
    const TileView t = tile_view(a.band, a.grid, tIdx);
    const int n = t.R * t.C;
    const uint8_t* packing = a.arena + a.offsets[tIdx];
    const uint32_t len = a.lens[tIdx];
    // CodecHuffman.decode header (CodecHuffman.java:134-143)
    const int pred = len >= 10 ? int(packing[1]) : 0;
    const int32_t seed = len >= 10 ? int32_t(load_le32(packing + 2)) : 0;
    const uint32_t nM32 = len >= 10 ? load_le32(packing + 6) : 0;
    const uint32_t expect = pred == G4_PRED_DIFF_NULLS ? uint32_t(n) : uint32_t(n - 1);
    if (len < 12 || pred < 1 || pred > 4 || nM32 < expect || nM32 > uint32_t(6 * n)) {
      if (tid == 0) a.status[tIdx] = G4_ERR_FORMAT;
      __syncthreads();
      continue;
    }
    const uint32_t delta = uint32_t(reinterpret_cast<uintptr_t>(packing) & 15u);
    const uint32_t span = len + delta;
    bool fast = pred == G4_PRED_TRIANGLE && span + 4u * kH2PadWords + 16u <= g.stageBytes && nM32 + 32u <= g.m32Cap &&
                nM32 <= kH2CompactChunk * uint32_t(NT) && t.C <= 2 * NT && size_t(kH2BandRows) * t.C * 4 <= g.stageBytes;
    int rc = 0;
    if (fast) {
      // stage: the packing from its 16-byte line start; whole 16-byte pieces by ONE bulk-async copy, the tail by bytes
      const uint8_t* src16 = packing - delta;
      const uint32_t nBulk = span & ~15u;
      if (tid == 0 && nBulk) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(nBulk) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(h2_smem_u32(sw)), "l"(src16),
                     "r"(nBulk), "r"(bar)
                     : "memory");
      }
      if (tid < 16 + 4 * kH2PadWords) {  // tail bytes and zero padding
        const uint32_t i = nBulk + uint32_t(tid);
        reinterpret_cast<uint8_t*>(sw)[i] = i < span ? src16[i] : uint8_t(0);
      }
      {  // the tree as huffman2_tree_kernel left it: kid, leafSym (adjacent in S) and the meta words
        const uint32_t* rec = reinterpret_cast<const uint32_t*>(trees + size_t(tIdx) * kH2TreeBytes);
        uint32_t* dstw = reinterpret_cast<uint32_t*>(&S.kid[0][0]);
        for (int i = tid; i < 768; i += NT) dstw[i] = __ldg(rec + i);
        if (tid < 4) reinterpret_cast<uint32_t*>(&S.tree)[tid] = __ldg(rec + 768 + tid);
      }
      if (nBulk) {
        uint32_t done = 0;
        while (!done)
          asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                       : "=r"(done)
                       : "r"(bar), "r"(parity)
                       : "memory");
        parity ^= 1u;
      }
      __syncthreads();
      const uint32_t nBits = span * 8u;
      if (S.tree.error == 2) fast = false;  // a tree deeper than the parser's path masks
      else if (S.tree.error) rc = 1;
      else if (S.tree.single >= 0) fast = false;  // one-symbol tree: no text in the stream
      else {
        h2_build_lut<NT>(S);
        rc = h2_decode_text<NT>(S, sw, nBits, S.tree.treeBits + 8u * delta, nM32, m32, g.m32Cap - 16u, spillArea, g.subBits, g.lookback);
        if (rc == 2) { fast = false; rc = 0; }
        else if (rc == 0) {
          uint2* exc = reinterpret_cast<uint2*>(S.mlut);  // the tables are dead once the text is decoded
          uint32_t nExc = 0;
          if (nM32 != uint32_t(n - 1)) {  // codes longer than one byte: one byte per residual + an exception list
            const int rc2 = h2_m32_compact<NT>(S, m32, nM32, uint32_t(n - 1), exc, spillArea);
            if (rc2 == 1) rc = 1;
            else if (rc2 == 2) fast = false;
            nExc = S.nExc;
          }
          if (rc == 0 && fast) h2_triangle_bytes<NT>(S, m32, seed, t, reinterpret_cast<int32_t*>(sw), exc, nExc);  // (ends with a barrier)
        }
      }
    }
    if (tid == 0) {
      if (!fast) defer[atomicAdd(deferCount, 1)] = tIdx;
      else a.status[tIdx] = rc ? G4_ERR_FORMAT : G4_OK;
    }
    __syncthreads();
  }
}

cudaError_t launch_huffman_encode(const EncodeArgs& a, int nCtas, cudaStream_t s) {
  static std::atomic<uint64_t> attr{0};
  cudaError_t ea = once_per_device(attr, [] {
    return cudaFuncSetAttribute(huffman_encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(sizeof(HuffEncShared)));
  });
  if (ea != cudaSuccess) return ea;
  huffman_encode_kernel<<<nCtas, kThreads, sizeof(HuffEncShared), s>>>(a);
  return cudaGetLastError();
}

template <int NT>
static cudaError_t launch_huffman2(const DecodeArgs& a, const Huff2Geom& g, size_t smem, int smCount, int nTilesUpper, uint32_t* spill,
                                   const uint8_t* trees, int* defer, int* deferCount, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(huffman2_decode_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  if (e != cudaSuccess) return e;
  int perSm = int((227u * 1024u) / (smem + 1024));
  const int cap = NT == 512 ? 2 : 4;
  if (perSm > cap) perSm = cap;
  if (perSm < 1) perSm = 1;
  int ctas = smCount * perSm;
  if (ctas > nTilesUpper) ctas = nTilesUpper;
  huffman2_decode_kernel<NT><<<ctas, NT, smem, s>>>(a, g, spill, trees, defer, deferCount);
  return cudaGetLastError();
}

size_t huffman2_spill_bytes(int smCount) { return size_t(smCount) * 4 * kH2MaxSub * kH2SpillWords * sizeof(uint32_t); }
size_t huffman2_tree_bytes(int nTiles) { return size_t(nTiles) * kH2TreeBytes; }

// fused: scratch of the fast path (spill of huffman2_spill_bytes, defer list of nTilesUpper ints, two zeroed counters)
cudaError_t launch_huffman_decode(const DecodeArgs& a, int nCtas, cudaStream_t s, const HuffFusedScratch& fused, int* launches) {
  // staging capacity of the fast decoder: 6 bits per sample of the tile (legacy Huffman over M32 bytes takes 4-5 bits
  // per sample on terrain), at most 160 KB (one CTA per SM)
  uint64_t bytes = uint64_t(a.band.tile_rows) * uint64_t(a.band.tile_cols) * 6 / 8 + 64;
  if (bytes > 160u * 1024u) bytes = 160u * 1024u;
  uint32_t stageWords = uint32_t((bytes + 3) / 4);
  if (stageWords < uint32_t(kHfStageWordsMin)) stageWords = kHfStageWordsMin;
  size_t smem = huff_fast_smem_bytes(stageWords);
  if (smem < sizeof(HuffDecShared)) smem = sizeof(HuffDecShared);
  static std::atomic<uint64_t> attr{0};
  cudaError_t ea = once_per_device(attr, [] {
    return cudaFuncSetAttribute(huffman_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                int(huff_fast_smem_bytes(160 * 1024 / 4 + 16)));
  });
  if (ea != cudaSuccess) return ea;
  DecodeArgs rest = a;
  if (a.band.elem_type == G4_ELEM_I32) {
    const uint32_t n = uint32_t(a.band.tile_rows) * uint32_t(a.band.tile_cols);
    Huff2Geom g;
    uint32_t stage = (n * 6u / 8u + 256u + 15u) & ~15u;
    const uint32_t bandBytes = uint32_t(kH2BandRows) * uint32_t(a.band.tile_cols) * 4u;
    if (stage < bandBytes) stage = (bandBytes + 15u) & ~15u;
    g.stageBytes = stage;
    g.m32Cap = (n + n / 16u + 48u + 15u) & ~15u;  // room for some codes longer than one byte
    g.subBits = kH2SubBits;
    g.lookback = kH2Lookback;
    const size_t smem2 = ((sizeof(Huff2Shared) + 127) & ~size_t(127)) + g.stageBytes + 16 + g.m32Cap;
    if (smem2 <= 112u * 1024u) {  // two 512-thread CTAs (or four 256-thread CTAs) per SM
      const int nTilesUpper = a.band.tiles_down * a.band.tiles_across;
      huffman2_tree_kernel<<<(nTilesUpper + 63) / 64, 64, 0, s>>>(a, fused.trees);
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) return e;
      e = n <= 16384u ? launch_huffman2<256>(a, g, smem2, fused.smCount, nTilesUpper, fused.spill, fused.trees, fused.defer, fused.counters, s)
                      : launch_huffman2<512>(a, g, smem2, fused.smCount, nTilesUpper, fused.spill, fused.trees, fused.defer, fused.counters, s);
      if (e != cudaSuccess) return e;
      *launches += 2;
      rest.list = fused.defer;
      rest.listCount = fused.counters;
      rest.counter = fused.counters + 1;
    }
  }
  huffman_decode_kernel<<<nCtas, kThreads, smem, s>>>(rest, stageWords);
  (*launches)++;
  return cudaGetLastError();
}

}  // namespace g4
