"""Times point reads from a GVRS file image resident on the GPU (GvrsDeviceImage.read_values, g4_decode_points) against the
paths users have without them, on the config-3 shard.

The shard (5,400 x 86,400 int32 synthetic terrain, 10,800 tiles of 180x240, codecs GvrsHuffman + GvrsDeflate + LSOP12) is
encoded on the GPU, written as a GVRS image with record checksums and made device resident (GvrsImage.to_device).  With CUDA
events, one warm-up call and --steps timed calls per row, the two rows of each comparison alternated call by call:
  1. one point                                         vs read_block(r, c, 1, 1)
  2. 10,000 points on a straight track, corner to corner vs read_raster(crop=False) + torch indexing
  3. 1,000,000 points inside a 4,096 x 4,096 block     vs read_block of that block + torch indexing
  4. 1,000,000 uniform random points (every tile)      vs read_raster(crop=False) + torch indexing
  5. 1,000 points read by a loop of single-cell read_block calls, the way available before read_values, vs one read_values.
Every result is checked to be identical to its comparison path first.  In a separate torch.profiler run per workload, the
share of kernel time spent in the mark, compact and store kernels is taken.  The card's name and power limit are read in
the same run and written with the numbers.

    python probes/bench_device_points.py --steps 7 --out result.json
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

POINT_KERNELS = ("point_mark_kernel", "point_compact_kernel", "point_store_kernel")


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
    # the point sets
    t = torch.linspace(0.0, 1.0, 10000, device=dev, dtype=torch.float64)
    track = ((t * (rows - 1)).round().long(), (t * (cols - 1)).round().long())
    br, bc, bn = 611, 20007, 4096
    in_block = (br + torch.randint(0, bn, (1 << 20,), device=dev, generator=gen), bc + torch.randint(0, bn, (1 << 20,), device=dev, generator=gen))
    uniform = (torch.randint(0, rows, (1 << 20,), device=dev, generator=gen), torch.randint(0, cols, (1 << 20,), device=dev, generator=gen))
    loop_pts = (torch.randint(0, rows, (1000,), device=dev, generator=gen), torch.randint(0, cols, (1000,), device=dev, generator=gen))
    one = (torch.tensor([2711], device=dev), torch.tensor([43210], device=dev))

    def whole(p):
        return lambda: dimg.read_raster(master)[p[0], p[1]]

    def block(p):
        return lambda: dimg.read_block(master, br, bc, bn, bn)[p[0] - br, p[1] - bc]

    loop_host = [(int(r), int(c)) for r, c in zip(loop_pts[0].tolist(), loop_pts[1].tolist())]

    def loop():
        return torch.cat([dimg.read_block(master, r, c, 1, 1).reshape(1) for r, c in loop_host])

    workloads = {
        "1 point": (one, lambda: dimg.read_block(master, 2711, 43210, 1, 1).reshape(1), "read_block(r, c, 1, 1)"),
        "10,000-point track, corner to corner": (track, whole(track), "read_raster(crop=False) + torch indexing"),
        "1,000,000 points in a 4,096 x 4,096 block": (in_block, block(in_block), "read_block(4096 x 4096) + torch indexing"),
        "1,000,000 uniform random points": (uniform, whole(uniform), "read_raster(crop=False) + torch indexing"),
        "1,000 points": (loop_pts, loop, "a loop of 1,000 read_block(r, c, 1, 1) calls"),
    }
    result_rows = {}
    for key, (pts, other, other_name) in workloads.items():
        ours_ms, other_ms = [], []
        for k in range(args.steps + 1):   # step 0 is the warm-up; the two rows alternate
            t_a, a = events(lambda: dimg.read_values(master, pts[0], pts[1]))
            k_tiles = int(dimg.lastTiles.numel())
            t_b, b = events(other)
            if k == 0:
                assert torch.equal(a, b), key
            else:
                ours_ms.append(t_a)
                other_ms.append(t_b)
            del a, b
        result_rows[key] = {"points": int(pts[0].numel()), "touched_tiles": k_tiles,
                            "read_values": {"ms_mean": float(np.mean(ours_ms)), "ms_all": ours_ms},
                            "comparison": {"path": other_name, "ms_mean": float(np.mean(other_ms)), "ms_all": other_ms},
                            "comparison_over_read_values": float(np.mean(other_ms) / np.mean(ours_ms)), "identical": True}

    from torch.profiler import ProfilerActivity, profile

    for key, (pts, _, _) in workloads.items():
        dimg.read_values(master, pts[0], pts[1])
        torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            dimg.read_values(master, pts[0], pts[1])
            torch.cuda.synchronize(dev)
        per, total = {k: 0.0 for k in POINT_KERNELS}, 0.0
        for e in prof.key_averages():
            us = float(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)))
            if "Memcpy" in e.key or "Memset" in e.key or us <= 0:
                continue
            total += us
            for k in POINT_KERNELS:
                if k in e.key:
                    per[k] += us
        result_rows[key]["profile"] = {"kernels_us": total, **{k + "_us": v for k, v in per.items()},
                                       "point_kernels_share": sum(per.values()) / total if total else None}

    result = {
        "what": "point reads of the config-3 shard (%d x %d int32, %d tiles of %dx%d, codecs %s, record checksums on) from a device "
                "resident GVRS image of %d bytes" % (rows, cols, n_tiles, tr, tc, "+".join(codecs), len(img.image)),
        "gpu": info, "steps": args.steps, "warmup": 1, "clock": "CUDA events on the read stream, rows alternated call by call",
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
