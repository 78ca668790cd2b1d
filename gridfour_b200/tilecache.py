"""Tile cache over a GVRS file image with BATCHED codec calls -- the caller north_star names for encodeTiles / decodeTiles.

Reference call pattern (paths under /root/reference/core/src/main/java/org/gridfour/gvrs/):
  RasterTileCache.getTile / readTileUsingAssistant  :113-179, :339-426   one tile per miss, LRU of GvrsCacheSize tiles
  TileDecompressionAssistant                        :50-275             a read-ahead thread that decompresses the next tile
  GvrsElement.readBlock / readValueInt              :298-404            loops over the cells of a block, tile by tile
  RasterTileCache.flush                             :286-294            writes every dirty tile, one codec call each
Here a block read first works out which tiles of the window are missing and decodes ALL of them with one
g4_decode_tile_list call, straight into their cache slots (each slot is its own small raster: the {offset, pitch} tile
references exist for exactly this); flush() encodes all dirty slots with one g4_encode_tile_list call.  The read-ahead
thread of the reference has no counterpart: a whole window costs one launch set.
Integer-coded float elements keep their int codes in the slots, as TileElementIntCodedFloat does; readBlockFloat /
writeBlockFloat map a block at the accessor with g4_icf_map."""
from collections import OrderedDict

import numpy as np

from ._lib import G4_DECLINED
from .gvrs import ELEM_FLOAT, ELEM_SHORT


class RasterTileCache:
    def __init__(self, image, master, element=0, max_tiles=16, verify=True):
        self.image, self.master, self.element = image, master, element
        spec = image.spec
        self.spec = spec
        e = spec.elements[element]
        if e.type_code == ELEM_SHORT:
            raise ValueError("short elements: use GvrsImage.read_raster (their widening pass works on a rectangle)")
        self.fill = e.fill_value
        self.icf = e.icf   # IntCodedFloat of an integer-coded float element, else None
        self.dtype = np.float32 if e.type_code == ELEM_FLOAT else np.int32
        self.R, self.C = spec.tile_rows, spec.tile_cols
        self.max_tiles = int(max_tiles)
        self.slots = np.empty((self.max_tiles, self.R, self.C), dtype=self.dtype)   # every slot = one tile's own raster
        self.resident = OrderedDict()   # tileIndex -> slot, least recently used first
        self.dirty = set()
        self.free = list(range(self.max_tiles))
        self.payload_off, self.lens, self.status = image.locate_payloads(master._context(), element, verify)
        self.arena = np.frombuffer(image.image, dtype=np.uint8)
        self.flushed = []   # (tile indices, TileBatch) of every flush(), for a writer
        self.decode_calls = self.encode_calls = 0

    # ---- residency ---------------------------------------------------------------------------------------------------
    def _evict_for(self, n):
        while len(self.free) < n:
            victims = [t for t in self.resident if t not in self._pinned]
            if not victims:
                raise RuntimeError("window larger than the cache")
            if any(t in self.dirty for t in victims[:n]):
                self.flush()
            t = victims[0]
            self.free.append(self.resident.pop(t))

    def fetch(self, tiles):
        """Makes `tiles` (at most max_tiles) resident; every missing one is decoded by ONE batched call."""
        tiles = list(dict.fromkeys(int(t) for t in tiles))
        if len(tiles) > self.max_tiles:
            raise ValueError("more tiles than cache slots")
        self._pinned = set(tiles)
        missing = [t for t in tiles if t not in self.resident]
        self._evict_for(len(missing))
        stored = []
        for t in missing:
            slot = self.free.pop()
            self.resident[t] = slot
            if self.status[t] == G4_DECLINED:     # a tile the file does not hold: RasterTile.setToNullState
                self.slots[slot][...] = self.fill
            else:
                stored.append(t)
        if stored:
            n = self.R * self.C
            refs = [(self.resident[t] * n, self.C) for t in stored]
            self.master.decodeTileList(self.arena, self.payload_off[stored], self.lens[stored], self.slots, refs, self.R, self.C)
            self.decode_calls += 1
        for t in tiles:
            self.resident.move_to_end(t)
        self._pinned = set()

    # ---- GvrsElement.readBlock (:298-404) / readValue -----------------------------------------------------------------
    def _windows(self, row, col, n_rows, n_cols):
        """The tiles a block touches, in chunks of at most max_tiles, each with the cell ranges to copy."""
        spec = self.spec
        if row < 0 or col < 0 or row + n_rows > spec.n_rows or col + n_cols > spec.n_cols or n_rows < 1 or n_cols < 1:
            raise ValueError("block outside the raster")
        tr0, tr1 = row // self.R, (row + n_rows - 1) // self.R
        tc0, tc1 = col // self.C, (col + n_cols - 1) // self.C
        tiles = [(tr, tc) for tr in range(tr0, tr1 + 1) for tc in range(tc0, tc1 + 1)]
        for k in range(0, len(tiles), self.max_tiles):
            yield tiles[k:k + self.max_tiles]

    def _span(self, tr, tc, row, col, n_rows, n_cols):
        r0, r1 = max(row, tr * self.R), min(row + n_rows, (tr + 1) * self.R)
        c0, c1 = max(col, tc * self.C), min(col + n_cols, (tc + 1) * self.C)
        return r0, r1, c0, c1

    def readBlock(self, row, col, nRows, nColumns):
        out = np.empty((nRows, nColumns), dtype=self.dtype)
        for chunk in self._windows(row, col, nRows, nColumns):
            self.fetch([tr * self.spec.tiles_across + tc for tr, tc in chunk])
            for tr, tc in chunk:
                r0, r1, c0, c1 = self._span(tr, tc, row, col, nRows, nColumns)
                tile = self.slots[self.resident[tr * self.spec.tiles_across + tc]]
                out[r0 - row:r1 - row, c0 - col:c1 - col] = tile[r0 - tr * self.R:r1 - tr * self.R, c0 - tc * self.C:c1 - tc * self.C]
        return out

    def readValue(self, row, col):
        return self.readBlock(row, col, 1, 1)[0, 0]

    def _icf(self):
        if self.icf is None:
            raise ValueError("readBlockFloat / writeBlockFloat: an integer-coded float element")
        return self.icf

    def readBlockFloat(self, row, col, nRows, nColumns):
        """The values of an integer-coded float element (float32): readBlock's codes mapped on the GPU."""
        icf = self._icf()
        return icf.to_float(self.readBlock(row, col, nRows, nColumns), context=self.master._context())

    def readValueFloat(self, row, col):
        return self.readBlockFloat(row, col, 1, 1)[0, 0]

    # ---- writes: GvrsElement.writeBlock / writeValue, RasterTileCache.flush (:286-294) -----------------------------------
    def writeBlock(self, row, col, block):
        block = np.asarray(block, dtype=self.dtype)
        n_rows, n_cols = block.shape
        for chunk in self._windows(row, col, n_rows, n_cols):
            self.fetch([tr * self.spec.tiles_across + tc for tr, tc in chunk])
            for tr, tc in chunk:
                t = tr * self.spec.tiles_across + tc
                r0, r1, c0, c1 = self._span(tr, tc, row, col, n_rows, n_cols)
                tile = self.slots[self.resident[t]]
                tile[r0 - tr * self.R:r1 - tr * self.R, c0 - tc * self.C:c1 - tc * self.C] = block[r0 - row:r1 - row, c0 - col:c1 - col]
                self.dirty.add(t)

    def writeValue(self, row, col, value):
        self.writeBlock(row, col, np.array([[value]], dtype=self.dtype))

    def writeBlockFloat(self, row, col, block):
        """Values of an integer-coded float element: mapped to codes on the GPU, then written as writeBlock does."""
        icf = self._icf()
        self.writeBlock(row, col, icf.to_int(np.asarray(block, dtype=np.float32), context=self.master._context()))

    def flush(self):
        """Encodes every dirty tile with ONE batched call (best-of over the codec list, raw fallback) and remembers the
        batch for a writer.  Returns (tile indices, TileBatch) or None when nothing was dirty."""
        if not self.dirty:
            return None
        tiles = sorted(self.dirty)
        n = self.R * self.C
        refs = [(self.resident[t] * n, self.C) for t in tiles]
        batch = self.master.encodeTileList(self.slots, refs, self.R, self.C)
        self.encode_calls += 1
        self.dirty.clear()
        self.flushed.append((tiles, batch))
        return tiles, batch
