/* CudaCodecLsop12.java -- drop-in for lsop/LsEncoder12.java + lsop/LsDecoder12.java behind the codec plugin API.  SOURCE ONLY.
 * The class lists both interfaces DIRECTLY because GvrsFileSpecification.addCompressionCodec inspects
 * getInterfaces() of the class itself (gvrs/GvrsFileSpecification.java:1608-1626); a public no-argument
 * constructor is invoked lazily by CodecHolder (gvrs/CodecHolder.java:189-234).
 */
package org.gridfour.cuda;

import org.gridfour.compress.ICompressionDecoder;
import org.gridfour.compress.ICompressionEncoder;

public class CudaCodecLsop12 extends CudaCodecBase implements ICompressionEncoder, ICompressionDecoder {

  private boolean deflateEnabled = true;         // LsEncoder12.java:78
  private boolean valueChecksumEnabled = false;

  public CudaCodecLsop12() {
    super(G4Native.CODEC_LSOP12);
  }

  /** LsEncoder12.setDeflateEnabled (lsop/LsEncoder12.java:93-119): false keeps every packing in the canonical-Huffman form. */
  public void setDeflateEnabled(boolean deflateEnabled) {
    this.deflateEnabled = deflateEnabled;
  }

  /** LsEncoder12.setValueChecksumEnabled (lsop/LsEncoder12.java:93-119): true stores the CRC-32C of the tile's values. */
  public void setValueChecksumEnabled(boolean valueChecksumEnabled) {
    this.valueChecksumEnabled = valueChecksumEnabled;
  }

  @Override
  int encodeId() {
    return G4Native.CODEC_LSOP12 | (deflateEnabled ? 0 : G4Native.LSOP12_NO_DEFLATE)
        | (valueChecksumEnabled ? G4Native.LSOP12_VALUE_CHECKSUM : 0);
  }
}
