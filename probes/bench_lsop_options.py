"""Times the LSOP12 encoder's two options (LsEncoder12.setDeflateEnabled / setValueChecksumEnabled) on the config-2 raster
and on the config-3 shard, and the decode cost of the value checksum.

  - config 2: 4,320 x 8,640 int32 synthetic terrain (g4_fill_terrain), 90 x 120 tiles, codec list [LSOP12];
  - config 3: one GPU's shard, 5,400 x 86,400 int32 terrain, 180 x 240 tiles, codec list [GvrsHuffman, GvrsDeflate, LSOP12].
For each raster and each of the four option combinations (Deflate on/off x checksum off/on) the encode is timed with CUDA
events, device resident.  Then the config-3 batches encoded with the checksum off and on (Deflate on, the reference's
default) are decoded and timed: the difference is the cost of the decode's check kernel (lsop_value_checksum_kernel), which
runs only over tiles whose packing carries a checksum.  One warm-up step runs every measurement once; each of the K timed
steps then runs every measurement once, the combinations in an order rotated by one every step.  The rasters and arenas are
larger than the 126 MB L2.  Every decode is checked against the raster.  Reported per combination: encode ms (mean and all
steps), bits/sample, and the share of the LSOP12 packings in the batch that took the Deflate form (type 1).  The card's name
and power limit are read in the same run and written with the numbers.

    python probes/bench_lsop_options.py --steps 5 --out result.json
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

COMBOS = [(True, False), (True, True), (False, False), (False, True)]  # (deflate, checksum)


def combo_name(c):
    return "deflate_%s_checksum_%s" % ("on" if c[0] else "off", "on" if c[1] else "off")


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
    if args.steps < 2:
        raise SystemExit("--steps must be at least 2")

    import torch

    import gridfour_b200 as g4
    from gridfour_b200 import _lib

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = gpu_info(0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = g4.Context(0, stream.cuda_stream)

    def master_of(names, deflate, checksum):
        spec = g4.CodecSpecification(default=False)
        classes = {"GvrsHuffman": (g4.CodecHuffman,), "GvrsDeflate": (g4.CodecDeflate,), "LSOP12": (g4.LsEncoder12, g4.LsDecoder12)}
        for n in names:
            spec.addCompressionCodec(n, *classes[n])
        m = g4.CodecMaster(spec, ctx)
        m.getEncoder("LSOP12").setDeflateEnabled(deflate)
        m.getEncoder("LSOP12").setValueChecksumEnabled(checksum)
        return m

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        r = fn()
        e1.record(stream)
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1), r

    rasters = {
        "config2": dict(rows=4320, cols=8640, tr=90, tc=120, codecs=["LSOP12"]),
        "config3": dict(rows=5400, cols=86400, tr=180, tc=240, codecs=["GvrsHuffman", "GvrsDeflate", "LSOP12"]),
    }
    result = {"gpu": info, "steps": args.steps, "warmup": 1, "rasters": {}}
    for rname, r in rasters.items():
        grid = torch.empty((r["rows"], r["cols"]), dtype=torch.int32, device=dev)
        ctx.fill_terrain(grid.data_ptr(), _lib.G4_ELEM_I32, 0, 0, r["rows"], r["cols"])
        torch.cuda.synchronize(dev)
        masters = {c: master_of(r["codecs"], *c) for c in COMBOS}
        lsop_index = r["codecs"].index("LSOP12")
        enc_ms = {combo_name(c): [] for c in COMBOS}
        stats = {}
        batches = {}
        for step in range(args.steps + 1):  # step 0 is the warm-up
            for k in range(len(COMBOS)):
                c = COMBOS[(k + step) % len(COMBOS)]
                ms, b = timed(lambda: masters[c].encodeTiles(grid, r["tr"], r["tc"]))
                if step:
                    enc_ms[combo_name(c)].append(ms)
                batches[c] = b
        for c in COMBOS:
            b = batches[c]
            codec, pred = b.codec.cpu().numpy(), b.predictor.cpu().numpy()
            is_lsop = codec == lsop_index
            stats[combo_name(c)] = {
                "bits_per_sample": 8.0 * b.total_bytes / grid.numel(),
                "arena_bytes": int(b.total_bytes),
                "tiles": int(codec.size),
                "lsop12_tiles": int(is_lsop.sum()),
                "lsop12_deflate_form_share": float((is_lsop & (pred == 1)).sum() / max(1, int(is_lsop.sum()))),
            }
        entry = {"raster": "%dx%d int32 terrain, %dx%d tiles, codecs %s" % (r["rows"], r["cols"], r["tr"], r["tc"], "+".join(r["codecs"])),
                 "encode_ms_mean": {k: float(np.mean(v)) for k, v in enc_ms.items()}, "encode_ms_all": enc_ms, "batches": stats}
        if rname == "config3":
            # decode of the same raster's packings without and with value checksums (Deflate on, the default)
            out = torch.empty_like(grid)
            pair = {"checksum_off": (True, False), "checksum_on": (True, True)}
            dec_ms = {k: [] for k in pair}
            launches = {}
            for step in range(args.steps + 1):
                for k in (list(pair) if step % 2 == 0 else list(pair)[::-1]):
                    c = pair[k]
                    l0 = ctx.launch_count
                    ms, _ = timed(lambda: masters[c].decodeTiles(batches[c], out=out))
                    launches[k] = ctx.launch_count - l0
                    assert torch.equal(out, grid), k
                    assert not bool(masters[c].lastStatus.any()), k
                    if step:
                        dec_ms[k].append(ms)
            mean = {k: float(np.mean(v)) for k, v in dec_ms.items()}
            entry["decode_ms_mean"] = mean
            entry["decode_ms_all"] = dec_ms
            entry["decode_launches"] = launches
            entry["decode_checksum_cost_ms"] = mean["checksum_on"] - mean["checksum_off"]
        result["rasters"][rname] = entry
        del batches, masters, grid
        torch.cuda.empty_cache()
    print(json.dumps(result))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
