// g4_huff2.cuh -- CodecHuffman decode, fused fast path for sm_100a: the M32 bytes never leave shared memory.
//
// Reference (under /root/reference/core/src/main/java/org/gridfour/compress/): CodecHuffman.java:133-153 (decode),
// HuffmanDecoder.java:65-187 (tree + text), CodecM32.java:313-356 (one-byte codes), PredictorModelTriangle.java:160-198
// (decode).
//
// One CTA per tile, persistent.  The packing is staged into shared memory by ONE bulk-async copy (cp.async.bulk +
// mbarrier); the legacy Huffman tree is parsed by one thread, an 11-bit single + multi-symbol table is built by all; the
// text is decoded by self-synchronising sub-sequences whose counting pass also stages the symbol bytes (slots inside the
// destination buffer, a small L2-resident spill behind them), so that after the prefix sum of the counts the bytes are
// COPIED to their place instead of being decoded a second time (the scheme of the LSOP12 text kernel, g4_lsop_fast.cu).
// The common case -- Triangle predictor, every M32 code one byte long (nM32 == cells - 1) -- is then finished in place:
// the residual field F (F[0][0] = seed, row 0 / column 0 / interior residuals in their stream order) is turned into its
// 2-D inclusive prefix sum band by band: warps scan rows out of the byte buffer into a 32-row band of int32 in shared
// memory (which reuses the packing's staging area), then one thread per column adds the band to its running column sum
// and writes the raster rows, coalesced, exactly once.  Every other tile (another predictor, a multi-byte M32 code, a
// single-symbol tree, an oversized packing) is handed to huffman_decode_kernel through a defer list.
#pragma once
#include "g4_huff_fast.cuh"
#include "g4_predict.cuh"  // the M32 byte automaton (m32_byte_map / m32_compose / m32_apply)

namespace g4 {

constexpr int kH2MaxSub = 1024;
constexpr uint32_t kH2SubBits = 448;   // target sub-sequence size (one round of sub-sequences for a 180x240 tile in a 512-thread CTA)
constexpr uint32_t kH2Lookback = 192;  // the first pass starts this many bits before a sub-sequence limit (swept: 64 .. 320)
constexpr int kH2StageWords = 22;      // registers that carry a thread's staged symbol bytes across the barrier
constexpr int kH2SpillWords = 16;      // words behind every slot in the per-CTA global scratch
constexpr int kH2BandRows = 32;
constexpr int kH2PadWords = 16;        // zero words behind the staged packing (a long code may be walked past the end)
constexpr int kH2FlagBad = 1, kH2FlagOverflow = 2;
constexpr uint32_t kH2ExcCap = 1024;  // multi-byte residuals a tile may hold on the fast path ((index, value) pairs over the dead LUT)
constexpr uint32_t kH2CompactChunk = 88;  // M32 bytes per thread of h2_m32_compact

struct H2TreeMeta {
  uint32_t treeBits;
  int nLeaf, single, error;
};

struct Huff2Shared {
  uint32_t mlut[1 << kLutBits];  // up to 3 symbols per lookup: s1 | s2 << 8 | s3 << 16 | bits << 24 | n << 28
  uint16_t lut[1 << kLutBits];   // sym | len << 9; bit 15: code longer than the table, low 9 bits = tree node reached
  uint16_t kid[512][2];
  int16_t leafSym[512];
  uint32_t endpos[kH2MaxSub];
  uint32_t startv[kH2MaxSub];
  uint16_t cnt[kH2MaxSub];
  uint8_t flag[kH2MaxSub];
  uint32_t scan[33];
  uint32_t nExc;                 // residuals whose M32 code is longer than one byte (h2_m32_compact)
  H2TreeMeta tree;
};

// Per-tile record of the tree kernel (huffman2_tree_kernel): kid[512][2] (2048 B), leafSym[512] (1024 B), H2TreeMeta (16 B)
constexpr int kH2TreeBytes = 2048 + 1024 + 16;

struct Huff2Geom {
  uint32_t stageBytes;  // staging area of the packing (also holds the band of the Triangle pass)
  uint32_t m32Cap;      // byte buffer of the M32 codes
  // kH2SubBits / kH2Lookback, passed as kernel arguments: compiled in as constants, the kernel measured 0.2 % slower
  // (B200, 1000 W)
  uint32_t subBits;     // target sub-sequence size
  uint32_t lookback;    // the first pass starts this many bits before a sub-sequence limit
};

__device__ __forceinline__ uint32_t h2_smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

struct H2Cursor {  // register bit window over the staged words, position kept relative to a limit (see BitCursor)
  uint32_t lo, hi, used, next;
  int rem;
  __device__ __forceinline__ void init(const uint32_t* sw, uint32_t p, uint32_t limit) {
    const uint32_t i = p >> 5;
    lo = sw[i];
    hi = sw[i + 1];
    used = p & 31u;
    next = i + 2;
    rem = int(limit) - int(p);
  }
  __device__ __forceinline__ uint32_t peek() const { return __funnelshift_r(lo, hi, used); }
  __device__ __forceinline__ uint32_t pos(uint32_t limit) const { return uint32_t(int(limit) - rem); }
  __device__ __forceinline__ void skip(const uint32_t* sw, uint32_t n) {
    used += n;
    rem -= int(n);
    if (used >= 32u) {
      lo = hi;
      hi = sw[next++];
      used -= 32u;
    }
  }
};

// HuffmanDecoder.decodeTree (:65-161) over the staged words, bounds-checked.  One thread.
// Nodes are numbered in pre-order, so the LEFT child of branch n is n + 1 and only the right links are stored
// (kid[n][1]; kid[n][0] = n + 1 is written as well for the walkers).  The path from the root is kept in two register
// bit masks (expR: the node at that depth has its left subtree done; amR: the node at that depth is a right child), so
// the dependent chain of a token is a few shifts: the only shared-memory read (the parent's id, for the right link) feeds
// a store, not the control flow.  Depth is limited to 62; deeper trees set S.error = 2 (the caller defers the tile).
// Output: kid / leafSym (512 nodes each), pstack = 64 entries of scratch, meta = {treeBits (position after the tree, same
// origin as startBit), nLeaf, single symbol or -1, error}.  word(i) returns 32-bit word i of the bit stream.
template <class WordFn>
__device__ __forceinline__ void h2_parse_tree(uint16_t (*kid)[2], int16_t* leafSym, uint16_t* pstack, H2TreeMeta& M, WordFn word, uint32_t startBit,
                                              uint32_t nBits) {
  auto bits = [&](uint32_t pos, int n) {
    const uint32_t i = pos >> 5;
    return __funnelshift_r(word(i), word(i + 1), pos & 31u) & ((1u << n) - 1u);
  };
  M.error = 0;
  M.single = -1;
  if (startBit + 17 > nBits) { M.error = 1; return; }
  const int L = int(bits(startBit, 8)) + 1;
  M.nLeaf = L;
  uint32_t pos = startBit + 8;
  if (bits(pos, 1)) {
    M.single = int(bits(pos + 1, 8));
    M.treeBits = startBit + 17;
    return;
  }
  pos = startBit + 9;
  // register bit buffer with the next word fetched one refill ahead
  uint32_t wi = pos >> 5;
  uint64_t buf = ((uint64_t(word(wi + 1)) << 32) | word(wi)) >> (pos & 31u);
  int avail = 64 - int(pos & 31u);
  wi += 2;
  uint32_t nextWord = word(wi);
  uint64_t expR = 0, amR = 0;
  int depth = 0, nodes = 1, leaves = 0;
  bool done = false;
  int pendParent = -1, pendId = 0;
  leafSym[0] = -1;
  kid[0][0] = 1;
  pstack[0] = 0;  // node id at every depth of the current path
  while (leaves < L) {
    if (done || nodes >= 511 || pos + 9 > nBits + 8) { M.error = 1; return; }
    const uint32_t x = uint32_t(buf) & 0x1ffu;
    const int id = nodes++;
    const bool isRight = (expR >> depth) & 1ull;
    // the right link of the parent: its id is read now, the store waits until the next token so that the (local-memory)
    // read is not what the in-order pipeline stalls on
    if (pendParent >= 0) kid[pendParent][1] = uint16_t(pendId);
    pendParent = isRight ? int(pstack[depth]) : -1;
    pendId = id;
    int used;
    if (x & 1u) {
      leafSym[id] = int16_t((x >> 1) & 0xffu);
      used = 9;
      leaves++;
      if (!isRight) expR |= 1ull << depth;  // the parent now expects its right child
      else {
        // the parent is complete, and so is every ancestor that is itself a right child: climb to the first node that is a
        // left child (amR bit clear); its parent now expects the right child
        const uint64_t cand = ~amR & ((2ull << depth) - 1ull);  // bit 0 (the root) is always a candidate
        const int d = 63 - __clzll((long long)cand);
        if (d == 0) done = true;  // the root is complete
        else {
          depth = d - 1;
          expR |= 1ull << depth;
        }
      }
    } else {
      if (depth >= 61) { M.error = 2; return; }
      leafSym[id] = -1;
      kid[id][0] = uint16_t(id + 1);
      used = 1;
      depth++;
      pstack[depth] = uint16_t(id);
      const uint64_t bit = 1ull << depth;
      expR &= ~bit;
      amR = isRight ? (amR | bit) : (amR & ~bit);
    }
    buf >>= used;
    avail -= used;
    pos += uint32_t(used);
    if (avail < 32) {
      buf |= uint64_t(nextWord) << avail;
      avail += 32;
      nextWord = word(++wi);
    }
  }
  if (pendParent >= 0) kid[pendParent][1] = uint16_t(pendId);
  if (!done || pos > nBits) { M.error = 1; return; }
  M.treeBits = pos;
}

template <int NT>
__device__ inline void h2_build_lut(Huff2Shared& S) {
  for (int e = threadIdx.x; e < (1 << kLutBits); e += NT) {
    int n = 0, d = 0;
    uint16_t entry = 0;
    for (; d < kLutBits; d++) {
      n = S.kid[n][(e >> d) & 1];
      if (S.leafSym[n] >= 0) { entry = uint16_t(S.leafSym[n] | ((d + 1) << 9)); break; }
    }
    if (d == kLutBits) entry = uint16_t(0x8000u | n);
    S.lut[e] = entry;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < (1 << kLutBits); e += NT) {
    uint32_t used = 0, n = 0, syms = 0;
    while (n < 3) {
      const uint32_t x = S.lut[(uint32_t(e) >> used) & ((1u << kLutBits) - 1u)];
      const uint32_t len = (x >> 9) & 15u;
      if ((x & 0x8000u) || used + len > uint32_t(kLutBits)) break;
      syms |= (x & 0xffu) << (8 * n);
      used += len;
      n++;
    }
    S.mlut[e] = syms | (used << 24) | (n << 28);
  }
  __syncthreads();
}

// One symbol whose code is longer than the table: walk the tree from the node the table entry names.
__device__ __forceinline__ int h2_long_symbol(const Huff2Shared& S, const uint32_t* sw, uint32_t e, uint32_t p0, uint32_t* after) {
  int n = int(e & 0x1ffu);
  uint32_t p = p0 + uint32_t(kLutBits);
  while (S.leafSym[n] < 0) {
    n = S.kid[n][(sw[p >> 5] >> (p & 31u)) & 1u];
    p++;
  }
  *after = p;
  return S.leafSym[n];
}

// Decodes one sub-sequence: from `start` to the first symbol boundary at or after `limit` (<= nBits).  With STORE the
// symbol bytes go to slot[0 .. slotWords) (shared memory) and on to spill[0 .. kH2SpillWords) (global).
// Byte accumulator of the staging pass: the pending (< 4) bytes sit TOP-justified in `acc`, so that they and the (up to
// three) symbol bytes of a lookup are contiguous in the pair (acc, m): the next output word is one funnel shift left, the
// new accumulator one funnel shift right.  qc8 = 8 x pending bytes.
struct H2ByteAcc {
  uint32_t acc, qc8, w;
  __device__ __forceinline__ void init() { acc = 0; qc8 = 0; w = 0; }
  __device__ __forceinline__ void put(uint32_t out, uint32_t* slot, uint32_t slotWords, uint32_t* spill) {
    if (w < slotWords) slot[w] = out;
    else if (w - slotWords < uint32_t(kH2SpillWords)) spill[w - slotWords] = out;
    w++;
  }
  // m24: symbol bytes in the low bytes (byte 3 zero), n8 = 8 x their number (8, 16 or 24)
  __device__ __forceinline__ void append(uint32_t m24, uint32_t n8, uint32_t* slot, uint32_t slotWords, uint32_t* spill) {
    const uint32_t out = __funnelshift_l(acc, m24, qc8);
    acc = __funnelshift_r(acc, m24, n8);
    qc8 += n8;
    if (qc8 >= 32u) {
      put(out, slot, slotWords, spill);
      qc8 -= 32u;
    }
  }
  __device__ __forceinline__ void finish(uint32_t* slot, uint32_t slotWords, uint32_t* spill) {
    if (qc8) put(acc >> (32u - qc8), slot, slotWords, spill);
  }
};

struct H2PosCursor {  // two staged words and the absolute bit position; a refill is due when a skip crosses a word boundary
  uint32_t lo, hi, next, pos;
  __device__ __forceinline__ void init(const uint32_t* sw, uint32_t p) {
    const uint32_t i = p >> 5;
    lo = sw[i];
    hi = sw[i + 1];
    next = i + 2;
    pos = p;
  }
  __device__ __forceinline__ uint32_t peek() const { return __funnelshift_r(lo, hi, pos); }
  __device__ __forceinline__ void skip(const uint32_t* sw, uint32_t n) {
    const uint32_t np = pos + n;
    if ((np ^ pos) & 32u) {
      lo = hi;
      hi = sw[next++];
    }
    pos = np;
  }
};

template <bool STORE>
__device__ __forceinline__ void h2_sub(const Huff2Shared& S, const uint32_t* sw, uint32_t nBits, uint32_t start, uint32_t limit, uint32_t* slot,
                                       uint32_t slotWords, uint32_t* spill, uint32_t* endOut, uint32_t* cntOut, int* flagOut) {
  H2PosCursor cur;
  cur.init(sw, start);
  const int lastFull = int(limit) - kLutBits;  // the whole table window lies before the limit up to this position
  uint32_t c = 0, end;
  H2ByteAcc A;
  A.init();
  int flag = 0;
  for (;;) {
    if (int(cur.pos) <= lastFull) {  // every symbol coded inside the window is consumed
      const uint32_t m = S.mlut[cur.peek() & ((1u << kLutBits) - 1u)];
      const uint32_t n = m >> 28;
      if (n) {
        cur.skip(sw, (m >> 24) & 15u);
        c += n;
        if (STORE) A.append(m & 0xffffffu, (m >> 25) & 0x18u, slot, slotWords, spill);
        continue;
      }
    }
    if (cur.pos >= limit) { end = cur.pos; break; }
    const uint32_t e = S.lut[cur.peek() & ((1u << kLutBits) - 1u)];
    uint32_t byte;
    if (!(e & 0x8000u)) {
      cur.skip(sw, (e >> 9) & 15u);
      byte = e & 0xffu;
    } else {
      const uint32_t p0 = cur.pos;
      uint32_t after;
      byte = uint32_t(h2_long_symbol(S, sw, e, p0, &after));
      if (after > nBits + 32u * kH2PadWords - 64u) { flag |= kH2FlagBad; end = p0; break; }
      cur.init(sw, after);
    }
    c++;
    if (STORE) A.append(byte, 8u, slot, slotWords, spill);
  }
  if (STORE) {
    A.finish(slot, slotWords, spill);
    if (A.w > slotWords + uint32_t(kH2SpillWords)) flag |= kH2FlagOverflow;
  }
  *endOut = end;
  *cntOut = c;
  *flagOut = flag;
}

// Linear byte sink of the copy pass: a run starts at any byte; its head goes out byte by byte up to the next word, the
// rest as aligned words, the tail by bytes (neighbouring runs share words, never bytes).
struct H2ByteSink {
  uint8_t* base;
  uint32_t addr;  // word-aligned offset of queue byte 0
  int head, cnt;
  uint64_t q;
  __device__ __forceinline__ void begin(uint8_t* b, uint32_t o0) {
    base = b;
    head = int(o0 & 3u);
    addr = o0 & ~3u;
    cnt = head;
    q = 0;
  }
  __device__ __forceinline__ void push(uint32_t bytes, int n) {  // n = 1..4
    q |= uint64_t(bytes) << (8 * cnt);
    cnt += n;
    if (cnt >= 4) {
      if (head) {
        for (int i = head; i < 4; i++) base[addr + i] = uint8_t(q >> (8 * i));
        head = 0;
      } else *reinterpret_cast<uint32_t*>(base + addr) = uint32_t(q);
      q >>= 32;
      cnt -= 4;
      addr += 4;
    }
  }
  __device__ __forceinline__ void end() {
    for (int i = head; i < cnt; i++) base[addr + i] = uint8_t(q >> (8 * i));
  }
};

// Decodes the text (tables ready, text at staged bit T0, nBits = end of the packing) into out[0 .. nSym).  `out` is a
// 16-byte aligned shared-memory buffer of outCap bytes.  All NT threads call.
// Returns 0 = done, 1 = malformed stream, 2 = a sub-sequence outgrew slot + spill (the caller defers the tile).
template <int NT>
__device__ int h2_decode_text(Huff2Shared& S, const uint32_t* sw, uint32_t nBits, const uint32_t T0, uint32_t nSym, uint8_t* out,
                              uint32_t outCap, uint32_t* spillArea, uint32_t subBits, uint32_t lookbackBits) {
  constexpr int kRounds = kH2MaxSub / NT;
  const int tid = threadIdx.x;
  if (T0 > nBits) return 1;
  const uint32_t avail = nBits - T0;
  uint32_t rounds = (avail / subBits + NT - 1) / NT;
  if (rounds < 1u) rounds = 1u;
  if (rounds > uint32_t(kRounds)) rounds = kRounds;
  uint32_t B = (avail + rounds * NT - 1) / (rounds * NT);
  if (B < 96u) B = 96u;
  const int nSub = int((avail + B - 1) / B);
  if (nSub == 0) return nSym == 0 ? 0 : 1;
  const uint32_t perSub = uint32_t(kH2StageWords) / rounds;
  uint32_t slotWords = (outCap / uint32_t(nSub)) >> 2;
  if (slotWords > perSub) slotWords = perSub;
  uint32_t* const out32 = reinterpret_cast<uint32_t*>(out);
  // pass 0: only the END of every sub-sequence matters here, so start kH2Lookback bits before the limit and rely on
  // self-synchronisation (a wrong guess is repaired by the passes below; the result never depends on it)
#pragma unroll 1
  for (int i = tid; i < nSub; i += NT) {
    uint32_t limit = T0 + uint32_t(i + 1) * B;
    if (limit > nBits) limit = nBits;
    uint32_t from = T0 + uint32_t(i) * B;
    const uint32_t lookback = B >= 256u ? lookbackBits : (lookbackBits * 2u) / 3u;
    if (limit - from > lookback) from = limit - lookback;
    uint32_t e, c;
    int f;
    h2_sub<false>(S, sw, nBits, from, limit, nullptr, 0, nullptr, &e, &c, &f);
    S.endpos[i] = e;
    S.startv[i] = 0xffffffffu;  // forces the exact decode of every sub-sequence in the first pass below
  }
  // synchronisation passes: sub-sequence i must start where i-1 ended.  Reads of endpos[i-1] may see this pass's or the
  // previous pass's value (both are candidates); the loop ends only after a pass in which nothing was rewritten.
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
        h2_sub<true>(S, sw, nBits, ns, limit, out32 + size_t(i) * slotWords, slotWords, spillArea + size_t(i) * kH2SpillWords, &e, &c, &f);
        vend[i] = e;
        S.cnt[i] = uint16_t(c);
        S.flag[i] = uint8_t(f);
        any = true;
      }
    }
    if (!__syncthreads_or(any ? 1 : 0)) break;
  }
  // symbol offsets: thread tid owns sub-sequences tid*kRounds .. +kRounds-1 for the scan
  uint32_t mySum = 0;
  int myFlags = 0;
#pragma unroll
  for (int j = 0; j < kRounds; j++) {
    const int i = tid * kRounds + j;
    if (i < nSub) {
      mySum += S.cnt[i];
      myFlags |= S.flag[i];
    }
  }
  uint32_t total;
  const uint32_t ex = block_exclusive_scan<NT>(mySum, S.scan, &total);
  const int flags = __syncthreads_or(myFlags);
  if (total < nSym) return 1;  // text shorter than the header claims
  if (flags & kH2FlagOverflow) return 2;
  uint32_t* offv = S.endpos;  // end positions are no longer needed: the array now holds the first symbol index of every sub-sequence
  {
    uint32_t run = ex;
#pragma unroll
    for (int j = 0; j < kRounds; j++) {
      const int i = tid * kRounds + j;
      if (i < nSub) {
        offv[i] = run;
        run += S.cnt[i];
      }
    }
  }
  __syncthreads();
  // slots -> registers (every thread: sub-sequences tid, tid + NT, ...), barrier, registers -> their place in the buffer
  uint32_t r[kH2StageWords];
#pragma unroll
  for (int j = 0; j < kH2StageWords; j++) r[j] = 0;
  for (uint32_t s = 0; s < rounds; s++) {
    const int i = tid + int(s) * NT;
    if (i < nSub) {
      const uint32_t* slot = out32 + size_t(i) * slotWords;
#pragma unroll
      for (int j = 0; j < kH2StageWords; j++)
        if (uint32_t(j) >= s * perSub && uint32_t(j) < s * perSub + slotWords) r[j] = slot[uint32_t(j) - s * perSub];
    }
  }
  __syncthreads();
  bool bad = false;
  for (uint32_t s = 0; s < rounds; s++) {
    const int i = tid + int(s) * NT;
    if (i >= nSub) continue;
    const uint32_t o0 = offv[i];
    if (o0 >= nSym) continue;  // padding bits behind the text that decode to symbols
    uint32_t n = S.cnt[i];
    if (n > nSym - o0) n = nSym - o0;
    if (S.flag[i] & kH2FlagBad) bad = true;  // an invalid code inside the text proper
    if (n == 0) continue;
    H2ByteSink sink;
    sink.begin(out, o0);
#pragma unroll
    for (int j = 0; j < kH2StageWords; j++) {
      const uint32_t at = (uint32_t(j) - s * perSub) * 4u;  // byte position of word j inside this sub-sequence's slot
      if (uint32_t(j) >= s * perSub && uint32_t(j) < s * perSub + slotWords && at < n) {
        const uint32_t m = n - at;
        sink.push(m >= 4u ? r[j] : (r[j] & ((1u << (8 * m)) - 1u)), m >= 4u ? 4 : int(m));
      }
    }
    if (n > slotWords * 4u) {  // the tail this thread spilled in the staging pass
      const uint32_t* sp = spillArea + size_t(i) * kH2SpillWords;
      for (uint32_t at = slotWords * 4u; at < n; at += 4u) {
        const uint32_t wv = *sp++, m = n - at;
        sink.push(m >= 4u ? wv : (wv & ((1u << (8 * m)) - 1u)), m >= 4u ? 4 : int(m));
      }
    }
    sink.end();
  }
  return __syncthreads_or(bad ? 1 : 0) ? 1 : 0;
}

// Tiles with M32 codes longer than one byte (spikes in the terrain): the code bytes in m32[0 .. nM32) are rewritten IN PLACE
// into one byte per residual -- byte k = the one-byte code of residual k, or 0 for a residual with a longer code, whose value
// goes to exc[] as (k, value) -- so that the Triangle pass below can run unchanged and add the few long values afterwards.
// Code boundaries come from a prefix scan over the START / CONT byte automaton (CodecM32.java:327-356, g4_predict.cuh).
// tmp: NT * 24 words of global scratch (the bytes a thread produces wait there until every thread has read its chunk).
// All NT threads call.  Returns 0 = done, 1 = malformed stream, 2 = more long codes than exc[] holds (caller defers).
template <int NT>
__device__ __noinline__ int h2_m32_compact(Huff2Shared& S, uint8_t* m32, uint32_t nM32, uint32_t nVal, uint2* exc, uint32_t* tmp) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kW = NT / 32;
  const uint32_t chunk = (nM32 + NT - 1) / NT;  // <= kH2CompactChunk (checked by the caller)
  const uint32_t b0 = uint32_t(tid) * chunk < nM32 ? uint32_t(tid) * chunk : nM32;
  const uint32_t b1 = b0 + chunk < nM32 ? b0 + chunk : nM32;
  if (tid == 0) S.nExc = 0;
  uint32_t f = 2u;  // identity
  for (uint32_t b = b0; b < b1; b++) f = m32_compose(f, m32_byte_map(m32[b]));
  uint32_t inc = f;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc = m32_compose(y, inc);
  }
  __syncthreads();
  if (lane == 31) S.scan[warp] = inc;
  __syncthreads();
  uint32_t pre = 2u, all = 2u;
#pragma unroll
  for (int w = 0; w < kW; w++) {
    const uint32_t m = S.scan[w];
    if (w < warp) pre = m32_compose(pre, m);
    all = m32_compose(all, m);
  }
  uint32_t excl = __shfl_up_sync(0xffffffffu, inc, 1);
  if (lane == 0) excl = 2u;
  const uint32_t state0 = m32_apply(m32_compose(pre, excl), 0u);
  if (m32_apply(all, 0u) != 0u) return 1;  // (uniform) the stream ends inside a code
  uint32_t cnt = 0;
  {
    uint32_t st = state0;
    for (uint32_t b = b0; b < b1; b++) {
      if (st == 0u) cnt++;
      st = m32_apply(m32_byte_map(m32[b]), st);
    }
  }
  uint32_t total;
  const uint32_t k0 = block_exclusive_scan<NT>(cnt, S.scan, &total);
  if (total != nVal) return 1;  // (uniform)
  // my residual bytes -> scratch, long codes -> exception list
  bool bad = false;
  {
    uint32_t* out = tmp + size_t(tid) * 24u;
    uint32_t st = state0, k = k0, acc = 0, nb = 0, w = 0;
    for (uint32_t b = b0; b < b1; b++) {
      const uint32_t byte = m32[b];
      if (st == 0u) {
        uint32_t r = byte;
        if (byte == 0x7Fu || byte == 0x81u) {
          int32_t val;
          if (m32_decode_at(m32, b, nM32, &val) == 0) bad = true;
          const uint32_t slot = atomicAdd(&S.nExc, 1u);
          if (slot < kH2ExcCap) exc[slot] = make_uint2(k, uint32_t(val));
          r = 0u;
        }
        acc |= r << (8u * nb);
        if (++nb == 4u) {
          out[w++] = acc;
          acc = 0;
          nb = 0;
        }
        k++;
      }
      st = m32_apply(m32_byte_map(byte), st);
    }
    if (nb) out[w] = acc;
  }
  if (__syncthreads_or(bad ? 1 : 0)) return 1;  // (also: every thread has read its chunk of m32)
  if (cnt) {
    const uint32_t* in = tmp + size_t(tid) * 24u;
    H2ByteSink sink;
    sink.begin(m32, k0);
    for (uint32_t at = 0; at < cnt; at += 4u) {
      const uint32_t wv = in[at >> 2], m = cnt - at;
      sink.push(m >= 4u ? wv : (wv & ((1u << (8 * m)) - 1u)), m >= 4u ? 4 : int(m));
    }
    sink.end();
  }
  __syncthreads();
  return S.nExc > kH2ExcCap ? 2 : 0;
}

// Triangle predictor, every residual a one-byte M32 code: raster = 2-D inclusive prefix sum of the residual field.
// m32 = the nM32 = R*C - 1 code bytes in stream order (SURVEY A.5: row 0 from column 1, column 0 from row 1, interior
// row-major), readable from m32 - 4; band = kH2BandRows * C int32 of shared memory.  All NT threads call.
// Per band of 32 rows: (1) warps turn rows of bytes into row prefix sums (int32, band); (2) the column sums run over
// (4-column quad, 4-row group) tasks in two passes -- group totals, then every task starts from the running column sum
// plus the totals of the groups above it and writes its four rows as 16-byte pieces, whole rows coalesced.  The group
// totals and the running column sums live in the sub-sequence arrays of S, which the decode no longer needs.
template <int NT>
__device__ inline void h2_triangle_bytes(Huff2Shared& S, const uint8_t* m32, int32_t seed, const TileView& t, int32_t* band, const uint2* exc,
                                         uint32_t nExc) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kW = NT / 32;
  constexpr int kGroups = kH2BandRows / 4;
  const int R = t.R, C = t.C;
  const int Q = C >> 2;
  // quads: C a multiple of 4, 16-byte aligned raster rows, group totals (kGroups * Q int4) and two carries (2 * Q int4) fit S
  const bool quads = (C & 3) == 0 && (t.pitch & 3) == 0 && (reinterpret_cast<uintptr_t>(t.base) & 15) == 0 &&
                     size_t(kGroups) * Q * 16 <= sizeof(S.endpos) + sizeof(S.startv) && size_t(2) * Q * 16 <= sizeof(S.cnt) + sizeof(S.flag);
  int4* gsum = reinterpret_cast<int4*>(S.endpos);   // endpos and startv are adjacent
  int4* carry = reinterpret_cast<int4*>(S.cnt);     // cnt and flag are adjacent; two buffers of Q
  if (quads)
    for (int q = tid; q < 2 * Q; q += NT) carry[q] = make_int4(0, 0, 0, 0);
  uint32_t run0 = 0, run1 = 0;  // (general form) running column sums of columns tid and tid + NT
  auto value = [](uint32_t b) { return b == 0x80u ? uint32_t(INT32_MIN) : uint32_t(int32_t(int8_t(b))); };  // CodecM32.java:313-324
  int cb = 0;  // carry buffer in use
  for (int r0 = 0; r0 < R; r0 += kH2BandRows) {
    const int nr = R - r0 < kH2BandRows ? R - r0 : kH2BandRows;
    for (int i = warp; i < kH2BandRows; i += kW) {  // row scans: band[i][c] = F[r][0] + ... + F[r][c]; zeros below the tile
      const int r = r0 + i;
      if (i >= nr) {
        if (quads)
          for (int q = lane; q < Q; q += 32) reinterpret_cast<int4*>(band + size_t(i) * C)[q] = make_int4(0, 0, 0, 0);
        continue;
      }
      const int baseR = r == 0 ? 0 : (C + R - 2) + (r - 1) * (C - 1);  // stream index of F[r][1]
      const uint32_t f0 = r == 0 ? uint32_t(seed) : value(m32[C - 1 + (r - 1)]);
      uint32_t rowCarry = 0;
      for (int c0 = 0; c0 < C; c0 += 256) {
        const int c = c0 + 8 * lane;
        const int o = baseR + c - 1;  // stream index of element (r, c); -1 for c == 0
        const int a = o & ~3;
        uint32_t lo = 0, hi = 0;
        if (c < C) {
          const uint32_t w0 = *reinterpret_cast<const uint32_t*>(m32 + a), w1 = *reinterpret_cast<const uint32_t*>(m32 + a + 4),
                         w2 = *reinterpret_cast<const uint32_t*>(m32 + a + 8);
          const uint32_t sh = uint32_t(o & 3) * 8u;
          lo = __funnelshift_r(w0, w1, sh);
          hi = __funnelshift_r(w1, w2, sh);
        }
        uint32_t e[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
          const uint32_t word = j < 4 ? lo : hi;
          // sign-extended byte j: prmt with the sign-replicating selector nibbles (8 | byte index); __byte_perm masks that bit away
          asm("prmt.b32 %0, %1, %2, %3;" : "=r"(e[j]) : "r"(word), "r"(0u), "r"(0x8880u | (uint32_t(j & 3) * 0x1111u)));
        }
        // the INT_MIN code 0x80 (rare): patch by value
        if (__any_sync(0xffffffffu, (((lo ^ 0x80808080u) - 0x01010101u) & ~(lo ^ 0x80808080u) & 0x80808080u) != 0u ||
                                        (((hi ^ 0x80808080u) - 0x01010101u) & ~(hi ^ 0x80808080u) & 0x80808080u) != 0u)) {
#pragma unroll
          for (int j = 0; j < 8; j++) {
            const uint32_t b = ((j < 4 ? lo : hi) >> (8 * (j & 3))) & 0xffu;
            if (b == 0x80u) e[j] = uint32_t(INT32_MIN);
          }
        }
        if (c == 0) e[0] = f0;
        if (c + 8 > C) {
#pragma unroll
          for (int j = 0; j < 8; j++)
            if (c + j >= C) e[j] = 0u;
        }
        uint32_t loc = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) { loc += e[j]; e[j] = loc; }
        const uint32_t inc = warp_inclusive_scan(loc);
        const uint32_t base = rowCarry + inc - loc;
        rowCarry += __shfl_sync(0xffffffffu, inc, 31);
        int32_t* dst = band + size_t(i) * C + c;
        if (c + 8 <= C && (C & 3) == 0) {
          *reinterpret_cast<int4*>(dst) = make_int4(int32_t(e[0] + base), int32_t(e[1] + base), int32_t(e[2] + base), int32_t(e[3] + base));
          *reinterpret_cast<int4*>(dst + 4) = make_int4(int32_t(e[4] + base), int32_t(e[5] + base), int32_t(e[6] + base), int32_t(e[7] + base));
        } else {
#pragma unroll
          for (int j = 0; j < 8; j++)
            if (c + j < C) dst[j] = int32_t(e[j] + base);
        }
      }
    }
    __syncthreads();
    if (nExc) {  // (uniform) residuals with long M32 codes: their byte is 0, their value is added to the rest of their row now
      for (uint32_t e = uint32_t(warp); e < nExc; e += uint32_t(kW)) {
        const uint32_t k = exc[e].x, val = exc[e].y;
        int r, c;
        if (k < uint32_t(C - 1)) { r = 0; c = int(k) + 1; }
        else if (k < uint32_t(C + R - 2)) { r = int(k) - (C - 1) + 1; c = 0; }
        else {
          const uint32_t j = k - uint32_t(C + R - 2);
          r = 1 + int(j / uint32_t(C - 1));
          c = 1 + int(j % uint32_t(C - 1));
        }
        if (r >= r0 && r < r0 + nr)
          for (int cc = c + lane; cc < C; cc += 32) atomicAdd(reinterpret_cast<unsigned int*>(band + size_t(r - r0) * C + cc), val);
      }
      __syncthreads();
    }
    if (quads) {
      auto add4 = [](int4 a, int4 b) {
        return make_int4(int32_t(uint32_t(a.x) + uint32_t(b.x)), int32_t(uint32_t(a.y) + uint32_t(b.y)), int32_t(uint32_t(a.z) + uint32_t(b.z)),
                         int32_t(uint32_t(a.w) + uint32_t(b.w)));
      };
      const int nTasks = kGroups * Q;
      for (int task = tid; task < nTasks; task += NT) {  // pass 1: totals of every (group, quad)
        const int g = task / Q, q = task - g * Q;
        const int4* b = reinterpret_cast<const int4*>(band + size_t(4 * g) * C) + q;
        int4 s4 = b[0];
        s4 = add4(s4, b[Q]);
        s4 = add4(s4, b[2 * Q]);
        s4 = add4(s4, b[3 * Q]);
        gsum[task] = s4;
      }
      __syncthreads();
      for (int task = tid; task < nTasks; task += NT) {  // pass 2: running sums and the raster rows
        const int g = task / Q, q = task - g * Q;
        int4 run = carry[cb * Q + q];
        for (int gg = 0; gg < g; gg++) run = add4(run, gsum[gg * Q + q]);
        const int4* b = reinterpret_cast<const int4*>(band + size_t(4 * g) * C) + q;
        int4* o = reinterpret_cast<int4*>(t.row(r0 + 4 * g)) + q;
        const int64_t pitch4 = t.pitch >> 2;
#pragma unroll
        for (int i = 0; i < 4; i++) {
          run = add4(run, b[i * Q]);
          if (4 * g + i < nr) o[i * pitch4] = run;
        }
        if (g == kGroups - 1) carry[(cb ^ 1) * Q + q] = run;  // the column sums through this band (rows below the tile add zero)
      }
      cb ^= 1;
    } else {
      // general form: thread c adds the band's rows to its running sum and writes the raster, one row per step
      if (tid < C) {
        const int32_t* b = band + tid;
        int32_t* o = t.row(r0) + tid;
        for (int i = 0; i < nr; i++) {
          run0 += uint32_t(b[size_t(i) * C]);
          o[int64_t(i) * t.pitch] = int32_t(run0);
        }
      }
      if (tid + NT < C) {
        const int32_t* b = band + tid + NT;
        int32_t* o = t.row(r0) + tid + NT;
        for (int i = 0; i < nr; i++) {
          run1 += uint32_t(b[size_t(i) * C]);
          o[int64_t(i) * t.pitch] = int32_t(run1);
        }
      }
    }
    __syncthreads();
  }
}

}  // namespace g4
