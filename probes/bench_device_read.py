"""Times reads from a GVRS file image resident on the GPU (GvrsImage.to_device, GvrsDeviceImage.read_block / read_raster)
against the host read path, on the config-3 shard.

The shard (5,400 x 86,400 int32 synthetic terrain, 10,800 tiles of 180x240, codecs GvrsHuffman + GvrsDeflate + LSOP12) is
encoded on the GPU and written as a GVRS image with record checksums.  The script measures, in one run:
  1. today's path: GvrsImage.read_raster (host image in, numpy raster out) plus the H2D copy of the raster into a tensor
     (host clock around work that ends in a device synchronise);
  2. GvrsImage.to_device, paid once per image (host clock, synchronised);
  3. GvrsDeviceImage.read_raster(crop=False) and g4_decode_tiles_bounded over the same resident arrays into a tensor,
     alternated step by step (CUDA events);
  4. unaligned read_block calls of 1,000 x 1,000, 4,096 x 4,096 and a 2,048 x 86,400 strip (CUDA events), and, in a
     separate torch.profiler run, the share of each read's kernel time spent in the store pass (window_store_kernel);
  5. the same strip through RasterTileCache.readBlock (host clock), for contrast: every fetch uploads the image prefix.
Every device result is compared with the host read_raster first.  The image (~208 MB) and the raster (1.87 GB) are larger
than the 126 MB L2.  The card's name and power limit are read in the same run and written with the numbers.

    python probes/bench_device_read.py --steps 7 --out result.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

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
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.steps < 3 or args.host_reps < 2:
        raise SystemExit("--steps must be at least 3 and --host-reps at least 2")

    import torch

    import gridfour_b200 as g4
    from gridfour_b200 import _lib, gvrs
    from gridfour_b200._lib import G4_MEM_DEVICE

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info(0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = g4.Context(0, stream.cuda_stream)
    codecs = ["GvrsHuffman", "GvrsDeflate", "LSOP12"]
    spec = g4.CodecSpecification(default=False)
    spec.addCompressionCodec("GvrsHuffman", g4.CodecHuffman)
    spec.addCompressionCodec("GvrsDeflate", g4.CodecDeflate)
    spec.addCompressionCodec("LSOP12", g4.LsEncoder12, g4.LsDecoder12)
    master = g4.CodecMaster(spec, ctx)

    tr, tc, rows, cols = 180, 240, 5400, 86400
    z = torch.empty((rows, cols), dtype=torch.int32, device=dev)
    ctx.fill_terrain(z.data_ptr(), 0, 0, 0, rows, cols)
    batch = master.encodeTiles(z, tr, tc)
    torch.cuda.synchronize(dev)
    gspec = gvrs.GvrsSpec(rows, cols, tr, tc, [gvrs.ElementSpec.integer("z")], codecs, checksum=True)
    w = gvrs.GvrsWriter(gspec, uuid=bytes(range(16)), time_modified=1700000000000)
    for name, rid, typ, content, desc in gvrs.codec_metadata(codecs):
        w.add_metadata(name, rid, typ, content, desc)
    w.add_tile_records(ctx, batch.arena.cpu().numpy(), batch.offsets.cpu().numpy().astype(np.uint64), batch.lens.cpu().numpy().astype(np.uint32))
    img = gvrs.GvrsImage.parse(w.finish(ctx))
    del batch
    raw_bytes = 4 * rows * cols

    def host_clock(fn):
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize(dev)
        return 1000.0 * (time.perf_counter() - t0), r

    def events(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        r = fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1), r

    # 1. today's path
    host_ms, host = [], None
    for k in range(args.host_reps + 1):   # rep 0 is the warm-up
        t, out = host_clock(lambda: torch.from_numpy(img.read_raster(master)).to(dev))
        if k == 0:
            host = out.cpu().numpy()
            assert np.array_equal(host, z.cpu().numpy())
        else:
            host_ms.append(t)
        del out

    # 2. to_device
    to_dev_ms = []
    for k in range(args.host_reps + 1):
        t, dimg = host_clock(lambda: img.to_device(ctx))
        if k:
            to_dev_ms.append(t)

    # 3. whole raster: read_raster(crop=False) vs g4_decode_tiles_bounded on the same arrays, alternated
    band = master._band((rows, cols), np.int32, tr, tc)
    grid = torch.empty((rows, cols), dtype=torch.int32, device=dev)
    status = torch.empty(gspec.tiles_down * gspec.tiles_across, dtype=torch.int32, device=dev)
    L = _lib.lib()
    cl = master._native_list()

    def bounded():
        st = L.g4_decode_tiles_bounded(ctx._h, C.byref(cl), C.byref(band), G4_MEM_DEVICE, dimg.image.data_ptr(), int(dimg.image.numel()),
                                       dimg.payload_off[0].data_ptr(), dimg.lens[0].data_ptr(), grid.data_ptr(), status.data_ptr())
        _lib.check(st, "g4_decode_tiles_bounded")

    whole = {"read_raster": [], "decode_tiles_bounded": []}
    for k in range(args.steps + 1):
        t_r, out = events(lambda: dimg.read_raster(master))
        t_b, _ = events(bounded)
        if k == 0:
            assert torch.equal(out, z) and torch.equal(grid, z)
        else:
            whole["read_raster"].append(t_r)
            whole["decode_tiles_bounded"].append(t_b)
        del out

    # 4. unaligned blocks
    blocks = {"1000x1000": (317, 40123, 1000, 1000), "4096x4096": (611, 20007, 4096, 4096), "2048x86400 strip": (1111, 0, 2048, 86400)}
    block_ms, block_info = {}, {}
    for key, (r, c, n, m) in blocks.items():
        ts = []
        for k in range(args.steps + 1):
            t, out = events(lambda: dimg.read_block(master, r, c, n, m))
            if k == 0:
                assert np.array_equal(out.cpu().numpy(), host[r:r + n, c:c + m]), key
            else:
                ts.append(t)
            del out
        block_ms[key] = ts
        td = (r + n - 1) // tr - r // tr + 1
        ta = (c + m - 1) // tc - c // tc + 1
        block_info[key] = {"row": r, "col": c, "n_rows": n, "n_cols": m, "covering_tiles": td * ta,
                           "staging_bytes": 4 * td * tr * ta * tc, "cells_bytes": 4 * n * m}
    from torch.profiler import ProfilerActivity, profile

    store_share = {}
    for key, (r, c, n, m) in blocks.items():
        dimg.read_block(master, r, c, n, m)
        torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            dimg.read_block(master, r, c, n, m)
            torch.cuda.synchronize(dev)
        store = total = 0.0
        for e in prof.key_averages():
            t = float(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)))
            if "Memcpy" in e.key or "Memset" in e.key or t <= 0:
                continue
            total += t
            if "window_store_kernel" in e.key:
                store += t
        store_share[key] = {"store_us": store, "kernels_us": total, "share": store / total if total else None}

    # 5. the strip through the host tile cache
    r, c, n, m = blocks["2048x86400 strip"]
    cache_ms = []
    for k in range(2):
        cache = g4.RasterTileCache(img, master, max_tiles=1024)
        t, out = host_clock(lambda: cache.readBlock(r, c, n, m))
        if k == 0:
            assert np.array_equal(out, host[r:r + n, c:c + m])
        cache_ms.append(t)
        del cache, out

    mean = lambda v: float(np.mean(v))  # noqa: E731
    result = {
        "what": "reads of the config-3 shard (%d x %d int32, %d tiles of %dx%d, codecs %s, record checksums on) from a GVRS image of "
                "%d bytes" % (rows, cols, gspec.tiles_down * gspec.tiles_across, tr, tc, "+".join(codecs), len(img.image)),
        "gpu": info, "steps": args.steps, "host_reps": args.host_reps, "warmup": 1, "image_bytes": len(img.image), "raw_bytes": raw_bytes,
        "host_read_raster_plus_h2d": {"ms_mean": mean(host_ms), "ms_all": host_ms, "gbs_raw": raw_bytes / mean(host_ms) / 1e6,
                                      "clock": "host clock, synchronised"},
        "to_device": {"ms_mean": mean(to_dev_ms), "ms_all": to_dev_ms, "clock": "host clock, synchronised (upload, record check, CRC)"},
        "whole_raster": {k: {"ms_mean": mean(v), "ms_all": v, "gbs_raw": raw_bytes / mean(v) / 1e6} for k, v in whole.items()},
        "blocks": {k: {**block_info[k], "ms_mean": mean(v), "ms_all": v, "gbs_cells": block_info[k]["cells_bytes"] / mean(v) / 1e6,
                       "store_pass": store_share[k]} for k, v in block_ms.items()},
        "strip_via_host_tile_cache": {"ms_all": cache_ms, "ms_mean": mean(cache_ms), "max_tiles": 1024,
                                      "clock": "host clock; result is a host array"},
    }
    result["whole_raster"]["read_raster_over_bounded_time"] = result["whole_raster"]["read_raster"]["ms_mean"] / \
        result["whole_raster"]["decode_tiles_bounded"]["ms_mean"]
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
