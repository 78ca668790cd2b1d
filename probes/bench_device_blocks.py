"""Times batched block reads from a GVRS file image resident on the GPU (GvrsDeviceImage.read_blocks, g4_decode_blocks)
against the paths users have without them, on the config-3 shard.

The shard (5,400 x 86,400 int32 synthetic terrain, 10,800 tiles of 180x240, codecs GvrsHuffman + GvrsDeflate + LSOP12) is
encoded on the GPU, written as a GVRS image with record checksums and made device resident (GvrsImage.to_device).  With CUDA
events, one warm-up call and --steps timed calls per row, the rows of each workload alternated call by call:
  1. 1 block of 256 x 256                        vs read_block
  2. 256 random blocks of 256 x 256              vs a loop of read_block calls; read_values on a meshgrid of int64 indices;
  3. 4,096 random blocks of 64 x 64                 read_raster(crop=False) + a torch gather
  4. 16 random blocks of 2,048 x 2,048
  5. 432 tile-sized blocks (180 x 240) at tile origins   vs read_values on a meshgrid (the store's fully aligned path)
Every result is checked to be identical to each comparison path first.  The meshgrid index tensors are built before the
clock starts, and their size is reported.  In a separate torch.profiler run per workload, the kernel time of the mark,
compact and store kernels is taken, and the store pass's rate is stated as (4 staged bytes read + output bytes) per cell
over the store kernel's time.  The card's name and power limit are read in the same run and written with the numbers.

    python probes/bench_device_blocks.py --steps 7 --out result.json
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

BLOCK_KERNELS = ("point_mark_kernel", "point_compact_kernel", "block_store_kernel")
HBM_BYTES_PER_S = 7.7e12   # B200 data sheet, one GPU at up to 1,000 W


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
    if args.steps < 7:
        raise SystemExit("--steps must be at least 7")

    import torch

    import gridfour_b200 as g4
    from gridfour_b200 import gvrs

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
    del z
    gspec = gvrs.GvrsSpec(rows, cols, tr, tc, [gvrs.ElementSpec.integer("z")], codecs, checksum=True)
    w = gvrs.GvrsWriter(gspec, uuid=bytes(range(16)), time_modified=1700000000000)
    for name, rid, typ, content, desc in gvrs.codec_metadata(codecs):
        w.add_metadata(name, rid, typ, content, desc)
    w.add_tile_records(ctx, batch.arena.cpu().numpy(), batch.offsets.cpu().numpy().astype(np.uint64), batch.lens.cpu().numpy().astype(np.uint32))
    img = gvrs.GvrsImage.parse(w.finish(ctx))
    del batch
    dimg = img.to_device(ctx)
    n_tiles = gspec.tiles_down * gspec.tiles_across

    def events(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        r = fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1), r

    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)

    def random_blocks(n, h, w):
        return (torch.randint(0, rows - h + 1, (n,), device=dev, generator=gen),
                torch.randint(0, cols - w + 1, (n,), device=dev, generator=gen))

    origins = torch.arange(0, n_tiles, n_tiles // 432, device=dev)[:432]   # 432 tiles spread over the grid
    sets = {
        "1 block of 256 x 256": ((torch.tensor([2711], device=dev), torch.tensor([43210], device=dev)), 256, 256),
        "256 random blocks of 256 x 256": (random_blocks(256, 256, 256), 256, 256),
        "4,096 random blocks of 64 x 64": (random_blocks(4096, 64, 64), 64, 64),
        "16 random blocks of 2,048 x 2,048": (random_blocks(16, 2048, 2048), 2048, 2048),
        "432 tile-sized blocks (180 x 240) at tile origins": (((origins // gspec.tiles_across) * tr, (origins % gspec.tiles_across) * tc),
                                                             tr, tc),
    }

    def meshgrid(b, h, w):
        r = (b[0].long()[:, None, None] + torch.arange(h, device=dev)[None, :, None]).expand(-1, h, w).contiguous()
        c = (b[1].long()[:, None, None] + torch.arange(w, device=dev)[None, None, :]).expand(-1, h, w).contiguous()
        return r, c

    def loop(b, h, w):
        origins = list(zip(b[0].tolist(), b[1].tolist()))

        def run():
            out = torch.empty((len(origins), h, w), dtype=torch.int32, device=dev)
            for i, (r, c) in enumerate(origins):
                dimg.read_block(master, r, c, h, w, out=out[i])
            return out
        return run

    def gather(b, h, w):
        def run():
            full = dimg.read_raster(master)
            return full[b[0].long()[:, None, None] + torch.arange(h, device=dev)[None, :, None],
                        b[1].long()[:, None, None] + torch.arange(w, device=dev)[None, None, :]]
        return run

    result_rows = {}
    for key, (b, h, w) in sets.items():
        n = int(b[0].numel())
        comps = {}
        if n == 1:
            comps["read_block"] = lambda b=b, h=h, w=w: dimg.read_block(master, int(b[0][0]), int(b[1][0]), h, w).reshape(1, h, w)
        else:
            if not key.startswith("432"):
                comps["a loop of %d read_block calls" % n] = loop(b, h, w)
            mr, mc = meshgrid(b, h, w)
            comps["read_values on a meshgrid of int64 indices"] = lambda mr=mr, mc=mc: dimg.read_values(master, mr, mc)
            if not key.startswith("432"):
                comps["read_raster(crop=False) + torch gather"] = gather(b, h, w)
        ours_ms, other_ms = [], {k: [] for k in comps}
        for step in range(args.steps + 1):   # step 0 is the warm-up; the rows alternate call by call
            t_a, a = events(lambda: dimg.read_blocks(master, b[0], b[1], h, w))
            k_tiles = int(dimg.lastTiles.numel())
            if step:
                ours_ms.append(t_a)
            for name, fn in comps.items():
                t_b, x = events(fn)
                if step == 0:
                    assert torch.equal(a, x), (key, name)
                else:
                    other_ms[name].append(t_b)
                del x
            del a
        row = {"blocks": n, "block_rows": h, "block_cols": w, "cells": n * h * w, "covered_tiles": k_tiles,
               "read_blocks": {"ms_mean": float(np.mean(ours_ms)), "ms_all": ours_ms}, "comparisons": {}, "identical": True}
        for name, ms in other_ms.items():
            c = {"ms_mean": float(np.mean(ms)), "ms_all": ms, "over_read_blocks": float(np.mean(ms) / np.mean(ours_ms))}
            if name.startswith("read_values"):
                c["index_bytes"] = 2 * 8 * n * h * w
            row["comparisons"][name] = c
        result_rows[key] = row
        comps.clear()
        torch.cuda.empty_cache()

    from torch.profiler import ProfilerActivity, profile

    for key, (b, h, w) in sets.items():
        dimg.read_blocks(master, b[0], b[1], h, w)
        torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            dimg.read_blocks(master, b[0], b[1], h, w)
            torch.cuda.synchronize(dev)
        per, total = {k: 0.0 for k in BLOCK_KERNELS}, 0.0
        for e in prof.key_averages():
            us = float(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)))
            if "Memcpy" in e.key or "Memset" in e.key or us <= 0:
                continue
            total += us
            for k in BLOCK_KERNELS:
                if k in e.key:
                    per[k] += us
        cells = result_rows[key]["cells"]
        store_s = per["block_store_kernel"] * 1e-6
        rate = (4 + 4) * cells / store_s if store_s else None
        result_rows[key]["profile"] = {"kernels_us": total, **{k + "_us": v for k, v in per.items()},
                                       "block_kernels_share": sum(per.values()) / total if total else None,
                                       "store_bytes_per_s": rate, "store_share_of_7.7TB/s": rate / HBM_BYTES_PER_S if rate else None}

    result = {
        "what": "block reads of the config-3 shard (%d x %d int32, %d tiles of %dx%d, codecs %s, record checksums on) from a device "
                "resident GVRS image of %d bytes" % (rows, cols, n_tiles, tr, tc, "+".join(codecs), len(img.image)),
        "gpu": info, "steps": args.steps, "warmup": 1, "clock": "CUDA events on the read stream, rows alternated call by call",
        "store_rate": "(4 B staged read + 4 B int32 output) * cells / block_store_kernel time, against 7.7 TB/s",
        "workloads": result_rows,
    }
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
