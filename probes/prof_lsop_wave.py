"""Kernel times of the LSOP12 decode set on the config-3 shard (10,800 tiles of 180x240), from torch.profiler.

The shard is the seeded synthetic terrain of bench.py, encoded on the device with the config-3 codecs (LSOP12 wins every
tile).  After one warm-up decode, K decodes run under torch.profiler with CUDA activities; the result is the mean device
time per decode of every kernel whose name holds `lsop`.  The card's name and power limit are read in the same run and
written with the numbers.

    python probes/prof_lsop_wave.py --steps 10 --out result.json
"""
import argparse
import json
import os
import subprocess
import sys

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
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    import gridfour_b200 as g4

    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    ctx = g4.Context(0, stream.cuda_stream)
    spec = g4.CodecSpecification(default=False)
    for n, c in (("GvrsHuffman", g4.CodecHuffman), ("GvrsDeflate", g4.CodecDeflate)):
        spec.addCompressionCodec(n, c, c)
    spec.addCompressionCodec("LSOP12", g4.LsEncoder12, g4.LsDecoder12)
    master = g4.CodecMaster(spec, ctx)
    rows, cols, tr, tc = 5400, 86400, 180, 240
    grid = torch.empty((rows, cols), dtype=torch.int32, device=dev)
    ctx.fill_terrain(grid.data_ptr(), 0, 0, 0, rows, cols)
    torch.cuda.synchronize(dev)
    batch = master.encodeTiles(grid, tr, tc)
    out = torch.zeros_like(grid)
    master.decodeTiles(batch, out=out)
    torch.cuda.synchronize(dev)
    assert torch.equal(out, grid)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            master.decodeTiles(batch, out=out)
        torch.cuda.synchronize(dev)
    kernels = {}
    for e in prof.events():
        if e.device_type.name != "CUDA" or "lsop" not in e.name:
            continue
        name = e.name.split("(")[0].replace("void ", "").replace("g4::(anonymous namespace)::", "")
        k = kernels.setdefault(name, {"calls": 0, "total_us": 0.0})
        k["calls"] += 1
        k["total_us"] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    for k in kernels.values():
        k["ms_per_decode"] = round(k["total_us"] / args.steps / 1000.0, 4)
        k["total_us"] = round(k["total_us"], 1)
    res = {"what": "LSOP12 decode kernels on the config-3 shard (10,800 tiles of 180x240), torch.profiler, mean of %d decodes" % args.steps,
           "gpu": gpu_info(0), "kernels": kernels}
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
