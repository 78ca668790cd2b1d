"""Times GVRS writes from a CUDA tensor (GvrsWriter.add_raster with a tensor, g4_encode_window) against the host write
path, on the config-3 shard.

The shard is 5,400 x 86,400 int32 synthetic terrain in 10,800 tiles of 180 x 240, codecs GvrsHuffman + GvrsDeflate + LSOP12,
record checksums on.  The script measures, in one run:
  1. end to end: GvrsWriter.add_raster + finish from a numpy raster (today's path) and from the same raster in a CUDA
     tensor (host clock around synchronised work), with the bytes each path moves across PCIe; the two images must be
     identical;
  2. g4_encode_window against g4_encode_tiles on the tile-aligned shard, alternated step by step (CUDA events);
  3. the shard cut to 5,393 x 86,387 (partial edge tiles) through g4_encode_window (CUDA events), and in a separate
     torch.profiler run the kernel time of the load pass (window_load_kernel);
  4. g4_encode_tiles of the shard as int16 with this library and with the parent commit's library (--parent-lib), built
     side by side and alternated step by step (CUDA events); the outputs must be identical;
  5. the partial-edge raster as integer-coded float values (scale 10): g4_encode_window against g4_encode_tiles_icf on a
     padded copy, alternated (CUDA events), and in a profiler run the load pass against the map it stands in for;
  6. the device-to-host copy of the tile records (CUDA events).
The raster (1.87 GB) is larger than the 126 MB L2.  The card's name and power limit are read in the same run and written
with the numbers.

    python probes/bench_device_write.py --parent-lib /path/to/parent/libg4codec.so --steps 5 --out result.json
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


def kernel_us(prof, names):
    """Device time (us) of the kernels whose names contain any of `names`, and of every kernel, in a profiler run."""
    sel = total = 0.0
    for e in prof.key_averages():
        t = float(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)))
        if "Memcpy" in e.key or "Memset" in e.key or t <= 0:
            continue
        total += t
        if any(n in e.key for n in names):
            sel += t
    return sel, total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--parent-lib", required=True, help="libg4codec.so built from the parent commit (the int16 comparison)")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.steps < 3 or args.host_reps < 2:
        raise SystemExit("--steps must be at least 3 and --host-reps at least 2")

    import torch
    from torch.profiler import ProfilerActivity, profile

    import gridfour_b200 as g4
    from gridfour_b200 import _lib, gvrs
    from gridfour_b200._lib import G4_MEM_DEVICE, BandDesc, CodecList

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
    prow, pcol = 5393, 86387
    z = torch.empty((rows, cols), dtype=torch.int32, device=dev)
    ctx.fill_terrain(z.data_ptr(), 0, 0, 0, rows, cols)
    torch.cuda.synchronize(dev)
    fill = -(2 ** 31)

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

    def alternate(fns, check):
        ts = {k: [] for k in fns}
        for step in range(args.steps + 1):   # step 0 is the warm-up
            outs = {}
            for k, fn in fns.items():
                t, outs[k] = events(fn)
                if step:
                    ts[k].append(t)
            if step == 0:
                check(outs)
            del outs
        return ts

    def same_pair(k1, k2, what):
        def check(o):
            assert same(o[k1], o[k2]), what + ": outputs differ"
        return check

    def same(a, b):
        if a.total_bytes != b.total_bytes:
            return False
        if not torch.equal(a.arena[:a.total_bytes], b.arena[:b.total_bytes]):
            return False
        return all(torch.equal(x, y) for x, y in [(a.offsets, b.offsets), (a.lens, b.lens), (a.codec, b.codec), (a.predictor, b.predictor),
                                                  (a.status, b.status)])

    # 1. end to end
    gspec = gvrs.GvrsSpec(rows, cols, tr, tc, [gvrs.ElementSpec.integer("z", fill_value=fill)], codecs, checksum=True)
    z_host = z.cpu().numpy()

    def write(grid):
        w = gvrs.GvrsWriter(gspec, uuid=bytes(range(16)), time_modified=1700000000000)
        for name, rid, typ, content, desc in gvrs.codec_metadata(codecs):
            w.add_metadata(name, rid, typ, content, desc)
        batch = w.add_raster(master, grid)
        return w.finish(ctx), batch

    e2e = {"host_numpy": [], "device_tensor": []}
    images = {}
    for k in range(args.host_reps + 1):
        for key, grid in [("host_numpy", z_host), ("device_tensor", z)]:
            t, (image, batch) = host_clock(lambda: write(grid))
            if k == 0:
                images[key] = (image, int(batch.total_bytes))
            else:
                e2e[key].append(t)
            del image, batch
    assert images["host_numpy"][0] == images["device_tensor"][0], "device-written image differs from the host-written one"
    image_bytes = len(images["host_numpy"][0])
    payload_bytes = images["host_numpy"][1]
    n_tiles = gspec.tiles_down * gspec.tiles_across
    del images

    # 2. tile-aligned: g4_encode_window vs g4_encode_tiles
    aligned = alternate({"encode_window": lambda: master.encodeTiles(z, tr, tc, padValue=fill),
                         "encode_tiles": lambda: master.encodeTiles(z, tr, tc)},
                        same_pair("encode_window", "encode_tiles", "tile-aligned"))

    # 3. partial edges
    zp = z[:prow, :pcol]   # a slice of the shard: pitch 86,400
    zpad = torch.full((rows, cols), fill, dtype=torch.int32, device=dev)
    zpad[:prow, :pcol] = zp
    partial = alternate({"encode_window": lambda: master.encodeTiles(zp, tr, tc, padValue=fill),
                         "encode_tiles_padded_copy": lambda: master.encodeTiles(zpad, tr, tc)},
                        same_pair("encode_window", "encode_tiles_padded_copy", "partial edges"))
    del zpad

    # 4. int16 encode: this library vs the parent's, alternated
    z16 = torch.clamp(z // 8, -30000, 30000).to(torch.int16)
    z16[100:300, 1000:3000] = -9999   # a patch of fill values (nulls)

    def bind(L):
        L.g4_context_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
        L.g4_context_destroy.argtypes = [C.c_void_p]
        L.g4_encode_arena_bound.argtypes = [C.POINTER(BandDesc)]
        L.g4_encode_arena_bound.restype = C.c_uint64
        L.g4_encode_tiles.argtypes = [C.c_void_p, C.POINTER(CodecList), C.POINTER(BandDesc), C.c_int, C.c_void_p, C.c_void_p, C.c_uint64,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
        h = C.c_void_p()
        _lib.check(L.g4_context_create(0, C.c_void_p(stream.cuda_stream), C.byref(h)), "g4_context_create")
        return L, h

    libs = {"this": bind(C.CDLL(_lib.LIB_PATH)), "parent": bind(C.CDLL(os.path.abspath(args.parent_lib)))}
    band16 = master._band((rows, cols), np.int16, tr, tc, fillValue=-9999)
    cl = master._native_list()
    cap = int(libs["this"][0].g4_encode_arena_bound(C.byref(band16)))
    bufs = {k: [torch.empty(cap, dtype=torch.uint8, device=dev), torch.empty(n_tiles, dtype=torch.int64, device=dev)] +
            [torch.empty(n_tiles, dtype=d, device=dev) for d in (torch.int32, torch.uint8, torch.uint8, torch.int32)] for k in libs}

    def enc16(k):
        L, h = libs[k]
        a, o, ln, cd, pr, st = bufs[k]
        total = C.c_uint64(0)
        _lib.check(L.g4_encode_tiles(h, C.byref(cl), C.byref(band16), G4_MEM_DEVICE, z16.data_ptr(), a.data_ptr(), cap, o.data_ptr(),
                                     ln.data_ptr(), cd.data_ptr(), pr.data_ptr(), st.data_ptr(), C.byref(total)), "g4_encode_tiles")
        return total.value

    def check16(o):
        assert o["this"] == o["parent"], "int16 totals differ"
        assert all(torch.equal(x[:o["this"]] if j == 0 else x, y[:o["this"]] if j == 0 else y)
                   for j, (x, y) in enumerate(zip(bufs["this"], bufs["parent"]))), "int16 outputs differ"

    short = alternate({"this": lambda: enc16("this"), "parent": lambda: enc16("parent")}, check16)
    for L, h in libs.values():
        L.g4_context_destroy(h)
    del bufs, z16

    # 5. ICF values, partial edges: g4_encode_window vs g4_encode_tiles_icf on a padded copy
    icf = g4.IntCodedFloat(10.0)
    vals = torch.empty((rows, cols), dtype=torch.float32, device=dev)
    ctx.fill_terrain(vals.data_ptr(), 1, 0, 0, rows, cols)
    vp = vals[:prow, :pcol]
    vpad = torch.full((rows, cols), float("nan"), dtype=torch.float32, device=dev)
    vpad[:prow, :pcol] = vp
    icf_rows = alternate({"encode_window": lambda: master.encodeTiles(vp, tr, tc, icf=icf, padValue=float("nan")),
                          "encode_tiles_icf_padded_copy": lambda: master.encodeTiles(vpad, tr, tc, icf=icf)},
                         same_pair("encode_window", "encode_tiles_icf_padded_copy", "ICF"))
    # kernel times from ONE profiler session (a later session in the same process recorded no kernels): the int32 and ICF
    # load passes (window_load_kernel<0> / <2>) and the map of the padded ICF copy they stand in for
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        master.encodeTiles(zp, tr, tc, padValue=fill)
        master.encodeTiles(vp, tr, tc, icf=icf, padValue=float("nan"))
        master.encodeTiles(vpad, tr, tc, icf=icf)
        torch.cuda.synchronize(dev)
    load_us, _ = kernel_us(prof, ["window_load_kernel<0>"])
    icf_load_us, _ = kernel_us(prof, ["window_load_kernel<2>"])
    icf_map_us, _ = kernel_us(prof, ["icf_to_int_kernel"])
    partial_profile = {"window_load_kernel_us": load_us, "staging_bytes": 4 * rows * cols, "source_bytes": 4 * prow * pcol}
    del vals, vpad

    # 6. the device-to-host copy of the records
    batch = master.encodeTiles(z, tr, tc)
    recs, _pos = gvrs.pack_tile_records_device(ctx, batch, 4096, True)
    torch.cuda.synchronize(dev)
    d2h = []
    for k in range(args.steps + 1):
        t, _host = events(lambda: recs.cpu())
        if k:
            d2h.append(t)
    n_rec = int(recs.numel())
    del batch, recs

    mean = lambda v: float(np.mean(v))  # noqa: E731
    summ = lambda d: {k: {"ms_mean": mean(v), "ms_all": v} for k, v in d.items()}  # noqa: E731
    raster_bytes = 4 * rows * cols
    result = {
        "what": "GVRS writes of the config-3 shard (%d x %d int32, %d tiles of %dx%d, codecs %s, record checksums on)"
                % (rows, cols, n_tiles, tr, tc, "+".join(codecs)),
        "gpu": info, "steps": args.steps, "host_reps": args.host_reps, "warmup": 1,
        "end_to_end": {**summ(e2e), "clock": "host clock, synchronised; add_raster + finish", "image_bytes": image_bytes,
                       "payload_bytes": payload_bytes, "records_bytes": n_rec,
                       "pcie_bytes_host_numpy": {"raster_up": raster_bytes, "payloads_down": payload_bytes, "payloads_up": payload_bytes,
                                                 "records_down": n_rec},
                       "pcie_bytes_device_tensor": {"records_down": n_rec, "content_positions_down": 8 * n_tiles},
                       "images_identical": True},
        "tile_aligned": {**summ(aligned), "clock": "CUDA events", "outputs_identical": True},
        "partial_edges": {**summ(partial), "clock": "CUDA events", "outputs_identical": True, "n_rows": prow, "n_cols": pcol,
                          "source_pitch": cols, "profile": partial_profile},
        "int16_encode_tiles": {**summ(short), "clock": "CUDA events, alternated with the parent commit's library",
                               "outputs_identical": True},
        "icf_partial_edges": {**summ(icf_rows), "clock": "CUDA events", "outputs_identical": True, "scale": 10.0,
                              "profile": {"window_load_kernel_us": icf_load_us, "icf_to_int_kernel_us": icf_map_us}},
        "records_d2h": {"ms_mean": mean(d2h), "ms_all": d2h, "bytes": n_rec, "gbs": n_rec / mean(d2h) / 1e6,
                        "clock": "CUDA events around tensor.cpu() (pageable destination)"},
    }
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
