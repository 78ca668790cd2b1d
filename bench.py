#!/usr/bin/env python3
"""bench.py -- GVRS tile decode/encode throughput (BASELINE.json metric) on N B200s of one node.

Default workload (N=1 and per rank at N>1, weak scaling): the per-GPU shard of BASELINE.json config 3 --
30 tile rows x 360 tile columns = 10,800 tiles of 180x240 int32 samples (5,400 x 86,400 samples, 1.866 GB raw)
of the synthetic fractal terrain (include/g4terrain.h); rank r holds tile rows [30r, 30r+30) of the 240-row
global grid; codec list [GvrsHuffman, GvrsDeflate, LSOP12] with best-of selection (CodecMaster rule).
`--config 1|2|4|5` runs the other BASELINE.json configs (parity-test / report cases, not the headline line).

A step = one decode pass over the shard (the headline direction).  `value` = 4 B x samples / device time with the
compressed payloads resident in HBM; `e2e` = the same through g4_decode_tiles with HOST (pinned) buffers, H2D of
the payloads and D2H of the decoded raster inside the timed region.  Encode throughput of the same shard is
reported in `encode`.

--dump-outputs DIR: after the timed steps, writes what the last timed step returned to a caller of decodeTiles --
`raster.npy` (the decoded raster, or a fixed seeded sample of it) and `status.npy` (the per-tile status) -- as float64
(float32 for a float32 raster; both exact), one pair per rank at N>1.  All ranks together write at most DUMP_SAMPLES
raster samples (32 MiB) plus the tile statuses.  The inputs are the seeded synthetic terrain, so two builds run with the
same arguments can be compared file for file.  (The GPU arm only: --impl reference decodes a smaller sample.)

--steps K: K timed decode steps; the untimed per-kernel-timing passes and the e2e line run K decode passes as well
(the tile-record pack / unpack line is a fixed 1 + 3 passes of another operation).

Run __graft_entry__.build() first: bench.py loads the libraries it made instead of rebuilding them, writes only to
--dump-outputs, and caches no bytecode in the tree.

--impl reference: the reference's algorithm on the host cores.  The reference is Java and no JVM exists in this
image, so this arm times the C++ oracle (oracle/, a line-by-line restatement) with a tile thread pool over all host
cores on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as build() left it, __pycache__ included

ORACLE_IDS = {"GvrsHuffman": 0, "GvrsDeflate": 1, "GvrsFloat": 2, "GvrsCanonicalHuffman": 3, "LSOP12": 4}
GLOBAL_TILE_ROWS = 240  # config 3: 43200 / 180

# per-GPU workloads; `rows`/`cols` are the samples one GPU holds
CONFIGS = {
    1: dict(name="config1: int32 4320x8640 (GEBCO 5-arcmin shape), 90x120 tiles", rows=4320, cols=8640, tr=90, tc=120, dtype="int32",
            codecs=["GvrsHuffman", "GvrsDeflate"]),
    2: dict(name="config2: int32 4320x8640, 90x120 tiles, LSOP12 only", rows=4320, cols=8640, tr=90, tc=120, dtype="int32",
            codecs=["LSOP12"]),
    3: dict(name="config3 per-GPU shard: 10800 tiles of 180x240 int32 (5400 x 86400 samples)", rows=5400, cols=86400, tr=180, tc=240,
            dtype="int32", codecs=["GvrsHuffman", "GvrsDeflate", "LSOP12"]),
    4: dict(name="config4: float32 10800x21600 (ETOPO shape), 120x120 tiles, CodecFloat", rows=10800, cols=21600, tr=120, tc=120,
            dtype="float32", codecs=["GvrsFloat"]),
}
SWEEP_TILES = [(60, 60), (90, 120), (120, 120), (128, 128), (180, 240), (256, 256), (512, 512)]
SWEEP_GRID = (23040, 15360)  # rows = lcm of the tile heights, cols = 2 x lcm of the tile widths; 1.42 GB raw per GPU (11x the L2)
METRIC = "GVRS tile decode GB/s of raw samples (config 3 shard, 180x240 tiles)"
DUMP_SAMPLES = 1 << 22  # raster samples written by --dump-outputs over all ranks: 32 MiB as float64
DUMP_SEED = 20240601


def dump_outputs(path, raster, status, rank, world):
    """Writes the decoded raster and the per-tile status of one decodeTiles call to path/raster.npy and path/status.npy
    (per rank when world > 1).  Each rank writes its whole raster if it has at most DUMP_SAMPLES // world samples, else a
    seeded sample of that many positions drawn over its flat index."""
    import torch

    os.makedirs(path, exist_ok=True)
    flat = raster.reshape(-1)
    per_rank = DUMP_SAMPLES // world
    if flat.numel() > per_rank:
        idx = np.unique(np.random.default_rng(DUMP_SEED).integers(0, flat.numel(), per_rank, dtype=np.int64))
        values = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()
    else:
        values = raster.cpu().numpy()
    suffix = "_rank%d" % rank if world > 1 else ""
    np.save(os.path.join(path, "raster%s.npy" % suffix), values.astype(np.float32 if values.dtype == np.float32 else np.float64))
    np.save(os.path.join(path, "status%s.npy" % suffix), status.cpu().numpy().astype(np.float64))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def profiled_traffic():
    """DRAM bytes per decode launch set from the committed ncu capture (profiles/decode_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "decode_traffic.json")
    if os.path.exists(p):
        return json.load(open(p))
    return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def workload_string(cfg, codecs, missing=()):
    """config.workload of BOTH arms (the driver compares the strings)."""
    return "%s, codecs=%s%s" % (cfg["name"], "+".join(codecs), (" (not yet on the GPU: %s)" % "+".join(missing)) if missing else "")


def cpu_sample(cfg, threads, budget_s, oracle):
    """The bounded CPU sample of the workload: whole tile rows from the top of rank 0's shard, encoded ONCE by the oracle.
    The number of tile rows is grown until one decode pass takes about budget_s / 8 (or the shard is exhausted)."""
    ids = [ORACLE_IDS[c] for c in cfg["codecs"]]
    tr, tc = cfg["tr"], cfg["tc"]
    is_f = cfg["dtype"] == "float32"
    max_rows = cfg["rows"] // tr
    n_rows = 1
    while True:
        gen = oracle.terrain_f32 if is_f else oracle.terrain_i32
        grid = gen(0, 0, n_rows * tr, cfg["cols"], n_threads=threads)
        t0 = time.perf_counter()
        arena, slot, lens = oracle.encode_grid(ids, grid, tr, tc, n_threads=threads)
        t_enc = time.perf_counter() - t0
        off = (np.arange(lens.size) * slot).astype(np.uint64)
        t0 = time.perf_counter()
        out = oracle.decode_grid(ids, arena, off, lens, grid.shape[0], grid.shape[1], tr, tc, dtype=np.float32 if is_f else np.int32,
                                 n_threads=threads)
        t_dec = time.perf_counter() - t0
        assert np.array_equal(out.view(np.uint32), grid.view(np.uint32))
        if t_dec > budget_s / 8 or t_enc > budget_s / 6 or n_rows >= max_rows:
            break
        n_rows = min(max_rows, n_rows * 3)
    return dict(ids=ids, grid=grid, arena=arena, off=off, lens=lens, t_enc=t_enc, tiles=int(lens.size), tile_rows=n_rows)


def cpu_decode_pass(cfg, smp, threads, oracle):
    tr, tc = cfg["tr"], cfg["tc"]
    is_f = cfg["dtype"] == "float32"
    t0 = time.perf_counter()
    oracle.decode_grid(smp["ids"], smp["arena"], smp["off"], smp["lens"], smp["grid"].shape[0], smp["grid"].shape[1], tr, tc,
                       dtype=np.float32 if is_f else np.int32, n_threads=threads)
    return time.perf_counter() - t0


def cpu_arm(cfg, threads, budget_s, oracle):
    """Oracle decode (and encode) throughput on the bounded sample; used for cpu_baseline of our own arm."""
    smp = cpu_sample(cfg, threads, budget_s, oracle)
    t_dec = min(cpu_decode_pass(cfg, smp, threads, oracle) for _ in range(2))
    grid, lens = smp["grid"], smp["lens"]
    raw = grid.size * 4
    tr, tc = cfg["tr"], cfg["tc"]
    res = {"decode_gbs": raw / t_dec / 1e9, "encode_gbs": raw / smp["t_enc"] / 1e9, "tiles": smp["tiles"], "dec_s": t_dec,
           "enc_s": smp["t_enc"], "bits_per_sample": 8.0 * float(lens.sum()) / grid.size}
    if cfg["dtype"] != "float32":
        # input distribution check (SURVEY.md 8d): Triangle-predictor M32 stream of the sample's first tiles
        one_byte, total_codes, hist = 0, 0, np.zeros(256, np.int64)
        for k in range(min(smp["tiles"], 8)):
            n, _seed, m32 = oracle.predictor_encode(oracle.PRED_TRIANGLE, grid[:tr, k * tc:(k + 1) * tc])
            b = np.frombuffer(m32, np.uint8)
            hist += np.bincount(b, minlength=256)
            total_codes += tr * tc - 1
            one_byte += (tr * tc - 1) - int(((b == 0x7F) | (b == 0x81)).sum())
        p = hist[hist > 0] / hist.sum()
        res["input_stats"] = {"m32_one_byte_fraction": one_byte / max(1, total_codes),
                              "m32_byte_entropy_bits": float(-(p * np.log2(p)).sum())}
    return res


def run_reference(args, rank, cfg):
    """--impl reference: the reference's own CPU algorithm (C++ restatement: no JVM in this image) on all host threads.
    The sample is generated and ENCODED ONCE; every warm-up / timed step is one whole decode pass over it."""
    if rank != 0:
        return
    from oracle import g4oracle as oracle

    threads = oracle.hardware_threads()
    smp = cpu_sample(cfg, threads, 24.0, oracle)
    for _ in range(args.warmup):
        cpu_decode_pass(cfg, smp, threads, oracle)
    times = [cpu_decode_pass(cfg, smp, threads, oracle) for _ in range(args.steps)]
    raw = smp["grid"].size * 4
    v = raw * len(times) / sum(times) / 1e9
    sample = ("%d tiles of %dx%d = the first %d tile row(s) of rank 0's shard, encoded once; one step = one decode pass over "
              "them; C++ restatement of the Java reference (no JVM in this image), tile thread pool over %d threads") % (
                  smp["tiles"], cfg["tr"], cfg["tc"], smp["tile_rows"], threads)
    metric = METRIC if args.config == 3 else "GVRS tile decode GB/s of raw samples (%s)" % cfg["name"].split(":")[0]
    line = {
        "impl": "reference", "metric": metric, "value": v, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * sum(times) / max(1, len(times)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
        "config": {"workload": workload_string(cfg, cfg["codecs"])},
        "cpu_baseline": {"value": v, "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample,
                         "encode_value": raw / smp["t_enc"] / 1e9, "bits_per_sample": 8.0 * float(smp["lens"].sum()) / smp["grid"].size},
        "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def build_master(g4, L, cfg, ctx):
    codecs = [c for c in cfg["codecs"] if L.g4_codec_supported(ORACLE_IDS[c], 0) and L.g4_codec_supported(ORACLE_IDS[c], 1)]
    missing = [c for c in cfg["codecs"] if c not in codecs]
    spec = g4.CodecSpecification(default=False)
    std = {"GvrsHuffman": (g4.CodecHuffman, g4.CodecHuffman), "GvrsDeflate": (g4.CodecDeflate, g4.CodecDeflate),
           "GvrsFloat": (g4.CodecFloat, g4.CodecFloat), "GvrsCanonicalHuffman": (g4.CodecCanonHuffman, g4.CodecCanonHuffman),
           "LSOP12": (g4.LsEncoder12, g4.LsDecoder12)}
    for c in codecs:
        spec.addCompressionCodec(c, *std[c])
    return g4.CodecMaster(spec, ctx), codecs, missing


def run_sweep(args, torch, dist, g4, L, ctx, dev, stream, rank, world, barrier):
    """Config 5: decode-only GB/s per tile size on one fixed grid (all sizes divide it), config-3 codec list."""
    rows, cols = SWEEP_GRID
    grid = torch.empty((rows, cols), dtype=torch.int32, device=dev)
    ctx.fill_terrain(grid.data_ptr(), 0, rank * rows, 0, rows, cols)
    peak, peak_src = peaks()
    out = torch.empty_like(grid)
    sweep = []
    for tr, tc in SWEEP_TILES:
        cfg = dict(CONFIGS[3], tr=tr, tc=tc)
        master, codecs, _ = build_master(g4, L, cfg, ctx)
        batch = master.encodeTiles(grid, tr, tc)
        for _ in range(args.warmup):
            master.decodeTiles(batch, out=out)
        torch.cuda.synchronize(dev)
        assert torch.equal(out, grid), "decode does not reproduce the input raster (%dx%d)" % (tr, tc)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ctx.set_async(True)  # pipelined device calls, see the config-3 loop in main()
        e0.record(stream)
        for _ in range(args.steps):
            master.decodeTiles(batch, out=out)
        e1.record(stream)
        barrier()
        ctx.set_async(False)
        assert int((master.lastStatus != 0).sum()) == 0 and torch.equal(out, grid), "decode failed in the timed region (%dx%d)" % (tr, tc)
        t = torch.tensor([e0.elapsed_time(e1) / 1000.0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        lens = batch.lens.cpu().numpy().astype(np.int64)
        hist = np.bincount(batch.codec.cpu().numpy(), minlength=256)
        gbs = 4.0 * rows * cols * world * args.steps / float(t[0]) / 1e9
        bps = 8.0 * float(lens.sum()) / (rows * cols)
        sweep.append({"tile": "%dx%d" % (tr, tc), "decode_gbs": gbs, "ms_per_step": 1000.0 * float(t[0]) / args.steps,
                      "bits_per_sample": bps, "hbm_frac_per_gpu": (4.0 + bps / 8.0) / 4.0 * gbs / world / peak,
                      "tile_choice": {c: int(hist[k]) for k, c in enumerate(codecs)} | {"raw": int(hist[255])}})
    if args.dump_outputs:  # the last timed step is that of the last tile size
        dump_outputs(args.dump_outputs, out, master.lastStatus, rank, world)
    if rank == 0:
        best = max(sweep, key=lambda s: s["decode_gbs"])
        print(json.dumps({"metric": "GVRS tile decode GB/s of raw samples (config 5 tile-size sweep)", "value": best["decode_gbs"],
                          "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": best["ms_per_step"],
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                          "config": {"workload": "config5: decode-only tile-size sweep on %dx%d int32 per GPU, codecs=%s; value = best size (%s)" % (
                              rows, cols, "+".join(CONFIGS[3]["codecs"]), best["tile"]), "l2": "inputs larger than L2"},
                          "peak": peak, "peak_source": peak_src, "sweep": sweep}))


def bind_to_gpu_numa_node(local_rank):
    """Best effort: run this rank's host threads (and first-touch its pinned buffers) on the NUMA node of its GPU."""
    try:
        import torch

        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id if hasattr(torch.cuda.get_device_properties(local_rank), "pci_bus_id") else None
        q = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True,
                           text=True).stdout.strip().lower()
        bus = q[4:] if q.startswith("0000") and len(q) > 12 else q  # sysfs uses a 4-digit domain
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return {"numa_node": node, "bound": False}
        cpus = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        allowed = ids & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "bound": bool(allowed), "cpus": len(allowed)}
    except Exception as e:  # containers often hide the topology
        return {"numa_node": None, "bound": False, "why": type(e).__name__}


def gpu_topology():
    """CPU / NUMA affinity of every GPU as `nvidia-smi topo -m` reports it (rank 0 only): names the host links the e2e copies share."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        rows = {}
        for line in out.splitlines():
            f = line.split()
            if f and f[0].startswith("GPU") and f[0][3:].isdigit():
                tail = [x for x in f[1:] if not (x == "X" or x.startswith(("NV", "PIX", "PXB", "PHB", "NODE", "SYS")))]
                rows[f[0]] = " ".join(tail)  # what is left: CPU affinity, NUMA affinity, GPU NUMA id
        return rows or None
    except Exception:
        return None


def measure_pcie(torch, dev, barrier, world, dist, nbytes=1 << 30):
    """Plain pinned-memory copies of 1 GiB per rank, ALL ranks at once: the platform's D2H / H2D ceiling that the e2e line
    (1.87 GB of decoded raster back to the host per step) runs into.  Returns GB/s per GPU (min over ranks)."""
    h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    res = {}
    for name, (dst, src) in {"d2h": (h, d), "h2d": (d, h)}.items():
        dst.copy_(src, non_blocking=True)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            dst.copy_(src, non_blocking=True)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) / 3000.0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[name + "_gbs_per_gpu"] = nbytes / float(t[0]) / 1e9
    del h, d
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", type=int, default=3, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--tile-rows", type=int, default=0, help="tile rows per GPU (default: the config's own)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--codecs", default="", help="comma-separated codec list instead of the config's own (e.g. GvrsHuffman: the "
                                                 "Huffman/Triangle half of the config-3 path on its own)")
    ap.add_argument("--strong", action="store_true",
                    help="config 3, strong scaling: the WHOLE 43200x86400 grid (240 tile rows) split over the ranks (N=1: one GPU holds it all)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the last step's decoded raster (sampled) and tile status to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; --impl reference decodes only a sample of the workload")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = dict(CONFIGS[3 if args.config == 5 else args.config])
    if args.codecs:
        cfg["codecs"] = [c for c in args.codecs.split(",") if c]
    if args.tile_rows:
        cfg["rows"] = args.tile_rows * cfg["tr"]
    if args.strong and args.config == 3:
        cfg["rows"] = (GLOBAL_TILE_ROWS // world) * cfg["tr"]
        cfg["name"] = "config3 strong scaling: 43200x86400 int32 over %d GPU(s), %d tiles of 180x240 per GPU" % (
            world, (GLOBAL_TILE_ROWS // world) * (cfg["cols"] // cfg["tc"]))
    if args.impl == "reference":
        run_reference(args, rank, cfg)
        return

    import torch
    import torch.distributed as dist

    import gridfour_b200 as g4
    from gridfour_b200 import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # the contract is ONE JSON line on stdout: NCCL prints its "NCCL version ..." banner to fd 1 when the communicator
        # is created, so fd 1 points at stderr while the process group comes up and the first collective runs
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    L = _lib.lib()
    # the context launches on torch's current stream so torch.cuda.Event brackets exactly the library's kernels
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx = g4.Context(local_rank, stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if args.config == 5:
        run_sweep(args, torch, dist, g4, L, ctx, dev, stream, rank, world, barrier)
        if world > 1:
            dist.destroy_process_group()
        return

    master, codecs, missing = build_master(g4, L, cfg, ctx)
    TILE_R, TILE_C = cfg["tr"], cfg["tc"]
    rows, cols = cfg["rows"], cfg["cols"]
    tile_rows = rows // TILE_R
    n_tiles = tile_rows * (cols // TILE_C)
    samples = rows * cols
    is_f = cfg["dtype"] == "float32"
    grid = torch.empty((rows, cols), dtype=torch.float32 if is_f else torch.int32, device=dev)
    if args.config == 3:
        # weak scaling: every rank holds one 30-tile-row band of the 240-tile-row global grid (rank r = band r at N = 8)
        bands = max(1, GLOBAL_TILE_ROWS // tile_rows)
        first_tile_row, _ = g4.shard_tile_rows(GLOBAL_TILE_ROWS, bands, rank % bands)
        row0 = first_tile_row * TILE_R
    else:
        row0 = rank * rows
    ctx.fill_terrain(grid.data_ptr(), 1 if is_f else 0, row0, 0, rows, cols)
    torch.cuda.synchronize(dev)

    # ---- encode (also produces the decode input) --------------------------------------------------------
    ctx.set_timing(True)
    enc_ms = []
    batch = None
    band_rows = 30 * TILE_R  # encode at most one config-3 shard at a time (bounds the candidate slots of the encoder)
    n_bands = (rows + band_rows - 1) // band_rows if (args.strong and rows > band_rows) else 1
    for i in range(3 if n_bands == 1 else 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        if n_bands == 1:
            batch = master.encodeTiles(grid, TILE_R, TILE_C)
        else:
            parts, base = [], 0
            for b in range(n_bands):
                pb = master.encodeTiles(grid[b * band_rows:(b + 1) * band_rows], TILE_R, TILE_C)
                used = (pb.total_bytes + 7) & ~7
                parts.append((pb.arena[:used].clone(), pb.offsets + base, pb.lens, pb.codec, pb.predictor, pb.status))
                base += used
                del pb
            band = master._band((rows, cols), np.int32, TILE_R, TILE_C)
            batch = g4.TileBatch(torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts]), torch.cat([p[2] for p in parts]),
                                 torch.cat([p[3] for p in parts]), torch.cat([p[4] for p in parts]), torch.cat([p[5] for p in parts]), base, band)
            del parts
        e1.record(stream)
        torch.cuda.synchronize(dev)
        enc_ms.append(e0.elapsed_time(e1))
    if len(enc_ms) == 1:
        enc_ms = enc_ms * 2
    enc_kernel_ms = {c: ctx.kernel_time_ms(1, ORACLE_IDS[c]) for c in codecs}
    lens = batch.lens.cpu().numpy().astype(np.int64)
    codec_of_tile = batch.codec.cpu().numpy()
    codec_hist = np.bincount(codec_of_tile, minlength=256)
    total_payload = int(lens.sum())
    bits_per_sample = 8.0 * total_payload / samples
    out = torch.zeros_like(grid)

    # ---- decode: device-resident, K timed steps ------------------------------------------------------------
    launches0 = ctx.launch_count
    for _ in range(args.warmup):
        master.decodeTiles(batch, out=out)
    torch.cuda.synchronize(dev)
    assert torch.equal(out.view(torch.int32), grid.view(torch.int32)), "decode does not reproduce the input raster"
    launches_per_step = (ctx.launch_count - launches0) // args.warmup
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # pipelined device calls (g4_context_set_async): a step only enqueues its kernels, as a tile cache that keeps several
    # windows in flight would; the per-tile status of every step is read after the timed region
    ctx.set_async(True)
    e0.record(stream)
    for _ in range(args.steps):  # the timed region: K decode passes, nothing else
        master.decodeTiles(batch, out=out)
    e1.record(stream)
    barrier()
    ctx.set_async(False)
    torch.cuda.synchronize(dev)
    assert int((master.lastStatus != 0).sum()) == 0, "a tile failed to decode in the timed region"
    assert torch.equal(out.view(torch.int32), grid.view(torch.int32)), "decode does not reproduce the input raster"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, master.lastStatus, rank, world)
    # per-kernel-set device time (CUDA events inside the library, on the launching stream): separate, untimed passes
    kernel_ms = {}
    for _ in range(args.steps):
        master.decodeTiles(batch, out=out)
        torch.cuda.synchronize(dev)
        for c in codecs:
            ms = ctx.kernel_time_ms(0, ORACLE_IDS[c])
            if ms is not None:
                kernel_ms.setdefault(c, []).append(ms)
    t_dec = e0.elapsed_time(e1) / 1000.0
    clocks = sampler.finish()
    t = torch.tensor([t_dec, float(np.mean(enc_ms[1:])) / 1000.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_dec, t_enc = float(t[0]), float(t[1])
    value = 4.0 * samples * world * args.steps / t_dec / 1e9
    enc_value = 4.0 * samples * world / t_enc / 1e9

    # ---- tile records either side of the path (SURVEY 8f row 1): framing + CRC-32C, then validation + CRC check ------
    records_info = None
    if not is_f:
        from gridfour_b200 import gvrs

        rec_ms = {"pack": [], "unpack": []}
        recs = pos = None
        for i in range(4):
            r0, r1, r2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            r0.record(stream)
            recs, pos = gvrs.pack_tile_records_device(ctx, batch, 4096, True)
            r1.record(stream)
            _off, _lens, st = gvrs.unpack_tile_records_device(ctx, recs, pos - 4096, True)
            r2.record(stream)
            torch.cuda.synchronize(dev)
            if i:
                rec_ms["pack"].append(r0.elapsed_time(r1))
                rec_ms["unpack"].append(r1.elapsed_time(r2))
        assert int((st != 0).sum()) == 0 and torch.equal(_lens.to(torch.int64), batch.lens.to(torch.int64))
        rb = int(recs.numel())
        records_info = {"record_bytes": rb, "pack_ms": float(np.mean(rec_ms["pack"])), "unpack_ms": float(np.mean(rec_ms["unpack"])),
                        "pack_gbs": rb / np.mean(rec_ms["pack"]) / 1e6, "unpack_gbs": rb / np.mean(rec_ms["unpack"]) / 1e6,
                        "what": "g4_pack_tile_records (frame + CRC-32C) / g4_unpack_tile_records (validate + CRC-32C) over the step's "
                                "payloads, device resident"}

    # ---- e2e: host buffers through the C ABI ------------------------------------------------------------------
    e2e = None
    if not args.no_e2e and samples * 4 <= (4 << 30):  # (a 15 GB pinned raster for the whole grid on one GPU is left out)
        h_arena = torch.empty(batch.total_bytes, dtype=torch.uint8).pin_memory()
        h_arena.copy_(batch.arena[: batch.total_bytes])
        h_off = batch.offsets.cpu().numpy().astype(np.uint64)
        h_len = batch.lens.cpu().numpy().astype(np.uint32)
        h_grid = torch.empty((rows, cols), dtype=grid.dtype).pin_memory()
        hb = g4.TileBatch(h_arena.numpy(), h_off, h_len, None, None, None, batch.total_bytes, batch.band)
        e2e_steps = args.steps
        master.decodeTiles(hb, out=h_grid.numpy())
        barrier()
        x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        x0.record(stream)
        for _ in range(e2e_steps):
            master.decodeTiles(hb, out=h_grid.numpy())  # H2D payloads, kernels, D2H raster: all on `stream`
        x1.record(stream)
        torch.cuda.synchronize(dev)
        t_e2e = x0.elapsed_time(x1) / 1000.0
        tt = torch.tensor([t_e2e], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        assert np.array_equal(h_grid.numpy()[:TILE_R].view(np.uint32), grid[:TILE_R].cpu().numpy().view(np.uint32))
        del h_grid, h_arena, hb
        pcie = measure_pcie(torch, dev, barrier, world, dist)
        e2e_total = 4.0 * samples * world * e2e_steps / float(tt[0]) / 1e9
        e2e = {"value": e2e_total, "unit": "GB/s",
               "h2d_bytes_per_step": int(batch.total_bytes + h_off.nbytes + h_len.nbytes),
               "d2h_bytes_per_step": int(samples * 4 + n_tiles * 4), "steps": e2e_steps,
               "per_gpu": e2e_total / world, "pcie_copy_peak": pcie, "frac_of_d2h_peak": e2e_total / world / pcie["d2h_gbs_per_gpu"],
               "host_binding": numa, "topology": gpu_topology() if rank == 0 else None,
               "note": "the decoded raster (4 B/sample) crossing PCIe bounds this line; pcie_copy_peak = plain pinned copies, all ranks at once"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant decode kernel set ------------------------------------------------------------
    peak, peak_src = peaks()
    dom = max(kernel_ms, key=lambda c: np.mean(kernel_ms[c])) if kernel_ms else None
    roofline = None
    if dom:
        kind = ORACLE_IDS[dom]
        idx = [k for k, c in enumerate(codecs) if c == dom][0]
        tiles_dom = int(codec_hist[idx])
        bytes_dom = int(lens[codec_of_tile == idx].sum())
        alg_bytes = 4.0 * tiles_dom * TILE_R * TILE_C + bytes_dom  # raw samples written once + payload read once
        ms = float(np.mean(kernel_ms[dom]))
        achieved = alg_bytes / (ms / 1000.0) / 1e9
        traffic = None
        tr_prof = profiled_traffic()
        if tr_prof and tr_prof.get("codec") == dom and args.config == 3 and not args.tile_rows:
            traffic = tr_prof["dram_bytes_per_launch_set"]
        roofline = {"bound": "hbm", "kernel": "%s decode (its kernels, bracketed by CUDA events on the launching stream)" % dom,
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                    "peak_source": peak_src, "kernel_ms": ms, "algorithmic_bytes_per_launch": alg_bytes, "kind": kind}
    # ---- CPU baseline (rank 0, N=1 only) ------------------------------------------------------------------------
    cpu = None
    if world == 1:
        from oracle import g4oracle as oracle

        threads = oracle.hardware_threads()
        ccfg = dict(cfg, codecs=codecs)
        r1 = cpu_arm(ccfg, 1, args.cpu_seconds / 3, oracle)
        rn = cpu_arm(ccfg, threads, args.cpu_seconds / 2, oracle)
        cpu = {"value": rn["decode_gbs"], "unit": "GB/s", "cores": threads, "kind": "port",
               "sample": "%d tiles of %dx%d from the workload's first tile row; oracle = C++ restatement of the Java reference "
                         "(no JVM in this image)" % (rn["tiles"], TILE_R, TILE_C),
               "single_thread_value": r1["decode_gbs"], "encode_value": rn["encode_gbs"],
               "encode_single_thread_value": r1["encode_gbs"], "bits_per_sample": rn["bits_per_sample"],
               "input_stats": rn.get("input_stats")}
    metric = METRIC if args.config == 3 else "GVRS tile decode GB/s of raw samples (%s)" % cfg["name"].split(":")[0]
    line = {
        "metric": metric, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * t_dec / args.steps, "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
        "dtype": cfg["dtype"], "data": "synthetic",
        "config": {"workload": workload_string(cfg, codecs, missing),
                   "l2": "inputs larger than L2 (payload %.0f MB + raster %.0f MB per step)" % (total_payload / 1e6, samples * 4 / 1e6),
                   "tile_choice": {c: int(codec_hist[k]) for k, c in enumerate(codecs)} | {"raw": int(codec_hist[255])}},
        "bits_per_sample": bits_per_sample,
        "encode": {"value": enc_value, "unit": "GB/s", "ms": 1000.0 * t_enc, "kernel_ms": enc_kernel_ms},
        "records": records_info,
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches_per_step * args.steps),
        "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
