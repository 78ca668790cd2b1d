"""Times integer-coded float (ICF) elements on the config-4 raster against config 4's CodecFloat path.

The raster is config 4's: 10,800 x 21,600 float32 synthetic terrain (g4_fill_terrain, decimetre-quantised), 120 x 120 tiles.
It is stored as ICF at scale 10, offset 0, with config 3's codec list [GvrsHuffman, GvrsDeflate, LSOP12], and as float32 with
CodecFloat (config 4 today).  Everything is device resident.  CUDA events time one warm-up step, then K steps in which
every measurement runs once, in the same order:
  - g4_icf_map in each direction alone, beside a cudaMemcpyAsync device-to-device copy of the same 933 MB (all three in
    GB/s of 8 bytes per sample: 4 read + 4 written);
  - g4_decode_tiles_icf, g4_decode_tiles of the same batch read as int32 codes, and CodecFloat decode of the floats;
  - g4_encode_tiles_icf and CodecFloat encode.
The raster and the arenas are larger than the 126 MB L2, so every pass reads from HBM.  The read-back is checked: every
decoded float must be within 1 ulp of the stored float; the number of cells that differ is reported.  The card's name and
power limit are read in the same run and written with the numbers.

    python probes/bench_icf.py --steps 5 --out result.json
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
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.steps < 3:
        raise SystemExit("--steps must be at least 3")

    import torch

    import gridfour_b200 as g4
    from gridfour_b200 import _lib

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info(0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = g4.Context(0, stream.cuda_stream)

    def master_of(names):
        spec = g4.CodecSpecification(default=False)
        classes = {"GvrsHuffman": (g4.CodecHuffman,), "GvrsDeflate": (g4.CodecDeflate,), "GvrsFloat": (g4.CodecFloat,),
                   "LSOP12": (g4.LsEncoder12, g4.LsDecoder12)}
        for n in names:
            spec.addCompressionCodec(n, *classes[n])
        return g4.CodecMaster(spec, ctx)

    icf_master = master_of(["GvrsHuffman", "GvrsDeflate", "LSOP12"])
    float_master = master_of(["GvrsFloat"])
    icf = g4.IntCodedFloat(10.0, 0.0)
    tr, tc, rows, cols = 120, 120, 10800, 21600
    n = rows * cols
    z = torch.empty((rows, cols), dtype=torch.float32, device=dev)
    ctx.fill_terrain(z.data_ptr(), _lib.G4_ELEM_F32, 0, 0, rows, cols)
    codes = torch.empty((rows, cols), dtype=torch.int32, device=dev)
    back = torch.empty_like(z)
    copy = torch.empty_like(z)
    out = torch.empty_like(z)
    out_i32 = torch.empty_like(codes)
    torch.cuda.synchronize(dev)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        r = fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1), r

    keys = ("map_to_int", "map_to_float", "memcpy_d2d", "decode_icf", "decode_i32", "decode_float", "encode_icf", "encode_float")
    ms = {k: [] for k in keys}
    check = {}
    for step in range(args.steps + 1):  # step 0 is the warm-up
        t = {}
        t["map_to_int"], _ = timed(lambda: icf.to_int(z, out=codes, context=ctx))
        t["map_to_float"], _ = timed(lambda: icf.to_float(codes, out=back, context=ctx))
        t["memcpy_d2d"], _ = timed(lambda: copy.copy_(z))
        t["encode_icf"], bi = timed(lambda: icf_master.encodeTiles(z, tr, tc, icf=icf))
        t["encode_float"], bf = timed(lambda: float_master.encodeTiles(z, tr, tc))
        as_i32 = g4.TileBatch(bi.arena, bi.offsets, bi.lens, None, None, None, bi.total_bytes, icf_master._band((rows, cols), np.int32, tr, tc))
        t["decode_icf"], _ = timed(lambda: icf_master.decodeTiles(bi, out=out))
        ok_icf = torch.equal(out.view(torch.int32), back.view(torch.int32))
        t["decode_i32"], _ = timed(lambda: icf_master.decodeTiles(as_i32, out=out_i32))
        ok_i32 = torch.equal(out_i32, codes)
        t["decode_float"], _ = timed(lambda: float_master.decodeTiles(bf, out=copy))
        ok_float = torch.equal(copy.view(torch.int32), z.view(torch.int32))
        assert ok_icf and ok_i32 and ok_float, (ok_icf, ok_i32, ok_float)
        if step == 0:
            assert not bool(torch.isnan(z).any())
            ulps = (out.view(torch.int32).to(torch.int64) - z.view(torch.int32).to(torch.int64)).abs()
            max_ulp = int(ulps.max())
            assert max_ulp <= 1, max_ulp
            check = {"max_ulp_read_back_vs_stored": max_ulp, "cells_differing_by_1_ulp": int((ulps == 1).sum()), "cells": n,
                     "codes_min": int(codes.min()), "codes_max": int(codes.max()),
                     "bits_per_sample_icf": 8.0 * bi.total_bytes / n, "bits_per_sample_float": 8.0 * bf.total_bytes / n,
                     "arena_bytes_icf": int(bi.total_bytes), "arena_bytes_float": int(bf.total_bytes),
                     "launches_decode_icf_minus_i32": None}
            l0 = ctx.launch_count
            icf_master.decodeTiles(as_i32, out=out_i32)
            l1 = ctx.launch_count
            icf_master.decodeTiles(bi, out=out)
            l2 = ctx.launch_count
            torch.cuda.synchronize(dev)
            check["launches_decode_icf_minus_i32"] = (l2 - l1) - (l1 - l0)
            continue
        for k in keys:
            ms[k].append(t[k])
    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    gbs = {k: 8.0 * n / mean[k] / 1e6 for k in ("map_to_int", "map_to_float", "memcpy_d2d")}
    raw = 4.0 * n
    gbs.update({k: raw / mean[k] / 1e6 for k in ("decode_icf", "decode_i32", "decode_float", "encode_icf", "encode_float")})
    result = {
        "what": "ICF (scale 10, offset 0; GvrsHuffman+GvrsDeflate+LSOP12) vs CodecFloat on the config-4 raster (%dx%d float32 terrain, "
                "%dx%d tiles), device resident, CUDA events per call; map/memcpy GB/s count 8 B/sample, codec GB/s count 4 B/sample "
                "of raw raster" % (rows, cols, tr, tc),
        "gpu": info, "steps": args.steps, "warmup": 1, **check,
        "ms_mean": mean, "ms_all": ms, "gbs": gbs,
        "map_over_memcpy_rate": {"to_int": gbs["map_to_int"] / gbs["memcpy_d2d"], "to_float": gbs["map_to_float"] / gbs["memcpy_d2d"]},
        "decode_icf_over_i32_time": mean["decode_icf"] / mean["decode_i32"],
        "decode_icf_over_float_rate": gbs["decode_icf"] / gbs["decode_float"],
        "encode_icf_over_float_rate": gbs["encode_icf"] / gbs["encode_float"],
    }
    print(json.dumps(result))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
