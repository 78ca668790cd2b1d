/* G4Native.java -- Panama FFM (java.lang.foreign, JDK 22+) binding of libg4codec.so (include/g4codec.h).
 *
 * SOURCE ONLY: no JDK exists in the build image, so this file has never been compiled there.  It shows the
 * binding a Gridfour maintainer adds; the same symbols are exercised from Python (gridfour_b200/_lib.py,
 * tests/test_abi.py), which is the tested binding.
 */
package org.gridfour.cuda;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.SymbolLookup;
import java.lang.invoke.MethodHandle;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

final class G4Native {

  static final int G4_OK = 0, G4_DECLINED = 1, G4_ERR_FORMAT = -2;
  static final int CODEC_HUFFMAN = 0, CODEC_DEFLATE = 1, CODEC_FLOAT = 2, CODEC_CANON_HUFFMAN = 3, CODEC_LSOP12 = 4;
  static final int LSOP12_NO_DEFLATE = 1 << 8, LSOP12_VALUE_CHECKSUM = 1 << 9;  // option bits of an LSOP12 codec id
  static final int MEM_HOST = 0;

  private static final Linker LINKER = Linker.nativeLinker();
  private static final SymbolLookup LIB =
    SymbolLookup.libraryLookup(System.getProperty("gridfour.cuda.library", "libg4codec.so"), Arena.global());

  private static MethodHandle h(String name, FunctionDescriptor fd) {
    return LINKER.downcallHandle(LIB.find(name).orElseThrow(), fd);
  }

  // int g4_context_create(int device, void* cuda_stream, g4_context** out)
  static final MethodHandle CONTEXT_CREATE = h("g4_context_create", FunctionDescriptor.of(JAVA_INT, JAVA_INT, ADDRESS, ADDRESS));
  static final MethodHandle CONTEXT_DESTROY = h("g4_context_destroy", FunctionDescriptor.ofVoid(ADDRESS));
  // int g4_encode_i32(ctx, codec_id, codec_index, n_rows, n_cols, const int32*, uint8* out, size_t cap, size_t* out_len, int* predictor)
  static final MethodHandle ENCODE_I32 = h("g4_encode_i32",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS));
  // int g4_decode_i32(ctx, codec_id, n_rows, n_cols, const uint8* packing, size_t len, int32* out)
  static final MethodHandle DECODE_I32 = h("g4_decode_i32",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS));
  static final MethodHandle ENCODE_F32 = h("g4_encode_f32",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS));
  static final MethodHandle DECODE_F32 = h("g4_decode_f32",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS));
  // int g4_encode_tiles(ctx, codecs, band, mem_space, grid, arena, arena_cap, offsets, lens, codec_out, predictor_out, status, total)
  static final MethodHandle ENCODE_TILES = h("g4_encode_tiles",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS,
      ADDRESS, ADDRESS, ADDRESS));
  // int g4_decode_tiles(ctx, codecs, band, mem_space, arena, offsets, lens, grid, status)
  static final MethodHandle DECODE_TILES = h("g4_decode_tiles",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, ADDRESS));

  // GVRS records (RecordManager.java:161-204,386-516; GridfourCRC32C.java): see include/g4codec.h
  // int g4_crc32c(ctx, mem_space, data, offsets, sizes, n, crc_out)
  static final MethodHandle CRC32C = h("g4_crc32c",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, ADDRESS));
  // uint64 g4_tile_records_bound(n_tiles, payload_bytes)
  static final MethodHandle TILE_RECORDS_BOUND = h("g4_tile_records_bound", FunctionDescriptor.of(JAVA_LONG, JAVA_INT, JAVA_LONG));
  // int g4_pack_tile_records(ctx, mem_space, arena, offsets, lens, tile_index, first_tile_index, n_tiles, checksum, base_pos,
  //                          records, records_cap, content_pos, total_bytes)
  static final MethodHandle PACK_TILE_RECORDS = h("g4_pack_tile_records",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, ADDRESS, ADDRESS, ADDRESS, JAVA_INT, JAVA_INT, JAVA_INT, JAVA_LONG,
      ADDRESS, JAVA_LONG, ADDRESS, ADDRESS));
  // int g4_unpack_tile_records(ctx, mem_space, image, image_len, content_pos, n_tiles, checksum, payload_offsets, lens, status)
  static final MethodHandle UNPACK_TILE_RECORDS = h("g4_unpack_tile_records",
    FunctionDescriptor.of(JAVA_INT, ADDRESS, JAVA_INT, ADDRESS, JAVA_LONG, ADDRESS, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, ADDRESS));

  /** One context (CUDA stream + scratch) per thread: decoder instances are entered concurrently by the
   *  application thread and the read-ahead thread (TileDecompressionAssistant.java:88). */
  static final ThreadLocal<MemorySegment> CONTEXT = ThreadLocal.withInitial(() -> {
    try (Arena a = Arena.ofConfined()) {
      MemorySegment out = a.allocate(ADDRESS);
      int rc = (int) CONTEXT_CREATE.invokeExact(Integer.getInteger("gridfour.cuda.device", 0), MemorySegment.NULL, out);
      if (rc != G4_OK) {
        throw new IllegalStateException("g4_context_create failed: " + rc + " (the CUDA codecs have no CPU fallback)");
      }
      return out.get(ADDRESS, 0);
    } catch (Throwable t) {
      throw new IllegalStateException(t);
    }
  });

  private G4Native() {
  }
}
