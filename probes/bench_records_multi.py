"""Times multi-element tile records against the one-element calls on the config-3 shard (10,800 tiles of 180x240).

Element 0 is the int32 synthetic terrain, element 1 the same terrain as int16 (it fits: |z| < 6,000).  Both are encoded
on the device with the config-3 codecs.  The script times, with CUDA events, one warm-up and then K steps that alternate:
  - g4_pack_tile_records / g4_unpack_tile_records of element 0 (what bench.py's `records` line measures),
  - g4_pack_tile_records_multi / g4_unpack_tile_records_multi of both elements,
  - g4_decode_tiles of element 1 from the multi-element image (payloads at any byte offset) and from its own encode arena
    (payloads 8-byte aligned).
Checksums are on.  The records are larger than the 126 MB L2, so every pass reads them from HBM.  The card's name and
power limit are read in the same run and written with the numbers.

    python probes/bench_records_multi.py --steps 7 --out result.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    name, power, clock = [x.strip() for x in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.steps < 5:
        raise SystemExit("--steps must be at least 5")

    import torch

    import gridfour_b200 as g4
    from gridfour_b200 import gvrs

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info(0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = g4.Context(0, stream.cuda_stream)
    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("GvrsHuffman", g4.CodecHuffman)
    spec.addCompressionCodec("GvrsDeflate", g4.CodecDeflate)
    spec.addCompressionCodec("LSOP12", g4.LsEncoder12, g4.LsDecoder12)
    master = g4.CodecMaster(spec, ctx)

    tr, tc, rows, cols = 180, 240, 5400, 86400
    z32 = torch.empty((rows, cols), dtype=torch.int32, device=dev)
    ctx.fill_terrain(z32.data_ptr(), 0, 0, 0, rows, cols)
    torch.cuda.synchronize(dev)
    assert int(z32.abs().max()) < 32767
    z16 = z32.to(torch.int16)
    b0 = master.encodeTiles(z32, tr, tc)
    b1 = master.encodeTiles(z16, tr, tc)
    torch.cuda.synchronize(dev)
    n = int(b0.lens.numel())
    band16 = master._band((rows, cols), np.int16, tr, tc)
    out16 = torch.empty_like(z16)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        r = fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1), r

    ms = {k: [] for k in ("pack_1", "unpack_1", "pack_multi", "unpack_multi", "decode_e1_image", "decode_e1_arena")}
    sizes = {}
    for step in range(args.steps + 1):  # step 0 is the warm-up
        t_p1, (rec1, pos1) = timed(lambda: gvrs.pack_tile_records_device(ctx, b0, 0, True))
        t_u1, (off1, len1, st1) = timed(lambda: gvrs.unpack_tile_records_device(ctx, rec1, pos1, True))
        t_pm, (recm, posm) = timed(lambda: gvrs.pack_tile_records_multi_device(ctx, [b0, b1], 0, True))
        t_um, (offm, lenm, stm) = timed(lambda: gvrs.unpack_tile_records_multi_device(ctx, recm, posm, 2, True))
        t_di, _ = timed(lambda: master.decodeTiles(g4.TileBatch(recm, offm[1], lenm[1], None, None, None, int(recm.numel()), band16), out=out16))
        ok_image = torch.equal(out16, z16)
        t_da, _ = timed(lambda: master.decodeTiles(b1, out=out16))
        ok_arena = torch.equal(out16, z16)
        if step == 0:
            assert int((st1 != 0).sum()) == 0 and int((stm != 0).sum()) == 0
            assert torch.equal(len1.to(torch.int64), b0.lens.to(torch.int64)) and torch.equal(lenm[0].to(torch.int64), b0.lens.to(torch.int64))
            assert torch.equal(lenm[1].to(torch.int64), b1.lens.to(torch.int64))
            assert ok_image and ok_arena
            sizes = {"record_bytes_1": int(rec1.numel()), "record_bytes_multi": int(recm.numel()),
                     "payload_bytes_e0": int(b0.lens.to(torch.int64).sum()), "payload_bytes_e1": int(b1.lens.to(torch.int64).sum()),
                     "e1_payloads_unaligned_in_image": int(((offm[1] & 7) != 0).sum())}
            continue
        for k, v in zip(ms, (t_p1, t_u1, t_pm, t_um, t_di, t_da)):
            ms[k].append(v)
    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    gbs = {"pack_1": sizes["record_bytes_1"] / mean["pack_1"] / 1e6, "unpack_1": sizes["record_bytes_1"] / mean["unpack_1"] / 1e6,
           "pack_multi": sizes["record_bytes_multi"] / mean["pack_multi"] / 1e6,
           "unpack_multi": sizes["record_bytes_multi"] / mean["unpack_multi"] / 1e6}
    result = {
        "what": "tile records of the config-3 shard (%d tiles of %dx%d; element 0 int32 terrain, element 1 the same terrain as int16; "
                "codecs GvrsHuffman+GvrsDeflate+LSOP12; checksums on), device resident, CUDA events per call" % (n, tr, tc),
        "gpu": info, "steps": args.steps, "warmup": 1, "n_tiles": n, **sizes,
        "ms_mean": mean, "ms_all": ms, "gbs_record_bytes": gbs,
        "multi_over_single_rate": {"pack": gbs["pack_multi"] / gbs["pack_1"], "unpack": gbs["unpack_multi"] / gbs["unpack_1"]},
        "decode_e1_image_over_arena_time": mean["decode_e1_image"] / mean["decode_e1_arena"],
    }
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
