/* CudaCodecBase.java -- shared implementation of the per-tile plugin calls over the C ABI.  SOURCE ONLY (no JDK in
 * the build image).  Mirrors ICompressionEncoder.java:61-91 / ICompressionDecoder.java:62-105 exactly:
 * encode returns null where the native call reports G4_DECLINED, decode throws IOException on G4_ERR_FORMAT.
 */
package org.gridfour.cuda;

import java.io.IOException;
import java.io.PrintStream;
import java.lang.foreign.Arena;
import java.lang.foreign.MemorySegment;

import static java.lang.foreign.ValueLayout.JAVA_BYTE;
import static java.lang.foreign.ValueLayout.JAVA_FLOAT;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

abstract class CudaCodecBase {

  private final int codecId;

  CudaCodecBase(int codecId) {
    this.codecId = codecId;
  }

  /** The codec id passed to g4_encode_i32: the plain id, with the option bits of an encoder that has options. */
  int encodeId() {
    return codecId;
  }

  public byte[] encode(int codecIndex, int nRows, int nCols, int[] values) {
    if (codecId == G4Native.CODEC_FLOAT) {
      throw new IllegalArgumentException("Integer encoding not supported");  // CodecFloat.java:116-125
    }
    try (Arena a = Arena.ofConfined()) {
      long cap = 6L * values.length + 1024;
      MemorySegment in = a.allocateFrom(JAVA_INT, values);
      MemorySegment out = a.allocate(cap);
      MemorySegment len = a.allocate(JAVA_LONG);
      int rc = (int) G4Native.ENCODE_I32.invokeExact(G4Native.CONTEXT.get(), encodeId(), codecIndex, nRows, nCols, in, out, cap, len,
        MemorySegment.NULL);
      if (rc == G4Native.G4_DECLINED) {
        return null;
      }
      if (rc != G4Native.G4_OK) {
        throw new IllegalStateException("g4_encode_i32: " + rc);
      }
      return out.asSlice(0, len.get(JAVA_LONG, 0)).toArray(JAVA_BYTE);
    } catch (RuntimeException e) {
      throw e;
    } catch (Throwable t) {
      throw new IllegalStateException(t);
    }
  }

  public byte[] encodeFloats(int codecIndex, int nRows, int nCols, float[] values) {
    if (codecId != G4Native.CODEC_FLOAT) {
      return null;  // CodecHuffman.java:241-244
    }
    try (Arena a = Arena.ofConfined()) {
      long cap = 6L * values.length + 4096;
      MemorySegment in = a.allocateFrom(JAVA_FLOAT, values);
      MemorySegment out = a.allocate(cap);
      MemorySegment len = a.allocate(JAVA_LONG);
      int rc = (int) G4Native.ENCODE_F32.invokeExact(G4Native.CONTEXT.get(), codecId, codecIndex, nRows, nCols, in, out, cap, len);
      if (rc == G4Native.G4_DECLINED) {
        return null;
      }
      if (rc != G4Native.G4_OK) {
        throw new IllegalStateException("g4_encode_f32: " + rc);
      }
      return out.asSlice(0, len.get(JAVA_LONG, 0)).toArray(JAVA_BYTE);
    } catch (RuntimeException e) {
      throw e;
    } catch (Throwable t) {
      throw new IllegalStateException(t);
    }
  }

  public int[] decode(int nRows, int nColumns, byte[] packing) throws IOException {
    try (Arena a = Arena.ofConfined()) {
      MemorySegment in = a.allocateFrom(JAVA_BYTE, packing);
      MemorySegment out = a.allocate(JAVA_INT, (long) nRows * nColumns);
      int rc = (int) G4Native.DECODE_I32.invokeExact(G4Native.CONTEXT.get(), codecId, nRows, nColumns, in, (long) packing.length, out);
      if (rc == G4Native.G4_DECLINED) {
        return null;
      }
      if (rc == G4Native.G4_ERR_FORMAT) {
        throw new IOException("Malformed packing");
      }
      if (rc != G4Native.G4_OK) {
        throw new IllegalStateException("g4_decode_i32: " + rc);
      }
      return out.toArray(JAVA_INT);
    } catch (IOException | RuntimeException e) {
      throw e;
    } catch (Throwable t) {
      throw new IllegalStateException(t);
    }
  }

  public float[] decodeFloats(int nRows, int nColumns, byte[] packing) throws IOException {
    if (codecId != G4Native.CODEC_FLOAT) {
      return null;
    }
    try (Arena a = Arena.ofConfined()) {
      MemorySegment in = a.allocateFrom(JAVA_BYTE, packing);
      MemorySegment out = a.allocate(JAVA_FLOAT, (long) nRows * nColumns);
      int rc = (int) G4Native.DECODE_F32.invokeExact(G4Native.CONTEXT.get(), codecId, nRows, nColumns, in, (long) packing.length, out);
      if (rc == G4Native.G4_ERR_FORMAT) {
        throw new IOException("Malformed packing");
      }
      if (rc != G4Native.G4_OK) {
        throw new IllegalStateException("g4_decode_f32: " + rc);
      }
      return out.toArray(JAVA_FLOAT);
    } catch (IOException | RuntimeException e) {
      throw e;
    } catch (Throwable t) {
      throw new IllegalStateException(t);
    }
  }

  public boolean implementsFloatingPointEncoding() {
    return codecId == G4Native.CODEC_FLOAT;
  }

  public boolean implementsIntegerEncoding() {
    return codecId != G4Native.CODEC_FLOAT;
  }

  public void analyze(int nRows, int nColumns, byte[] packing) throws IOException {
    // statistics stay with the reference's decoders (SURVEY.md 8f row 4)
  }

  public void reportAnalysisData(PrintStream ps, int nTilesInRaster) {
  }

  public void clearAnalysisData() {
  }
}
