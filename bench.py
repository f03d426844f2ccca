#!/usr/bin/env python
"""bench.py -- MPixels/s of the PNG decode hot path (inflate + unfilter) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm

A "step" decodes one batch of synthetic PNG image streams resident in HBM (value) or in pinned
host memory (e2e).  Workload (default): B x 7680x4320 RGBA8 "photo" images per GPU (SURVEY.md
section 8d corpus S0), compressed with zlib level 6 after the reference's filter rule.  Images
are independent, so ranks share nothing on the data path (weak scaling: B images per GPU).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (width, height, sixteen, default batch per GPU, default unique images)
    "8k-rgba8": (7680, 4320, False, 444, 8),
    "1080p-rgba8": (1920, 1080, False, 1184, 64),
    "8k-rgba16": (7680, 4320, True, 8, 8),
    "small": (512, 512, False, 64, 4),
}


_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly ONE JSON line: whatever libraries print there (NCCL's version banner ...) goes to
    stderr from now on; emit() writes the line to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: str):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (line + "\n").encode())


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="8k-rgba8", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (0 = workload default)")
    ap.add_argument("--unique", type=int, default=0, help="distinct images (0 = workload default)")
    ap.add_argument("--kind", default="photo", choices=["photo", "graphic", "noise"])
    ap.add_argument("--level", type=int, default=6, help="zlib level of the input streams")
    ap.add_argument("--encoder", default="zlib", choices=["zlib", "ref"],
                    help="who compresses the synthetic inputs: zlib (libpng-like streams, default) or 'ref' = "
                         "our GPU encoder at --encode-level, bit-identical to the reference's own output "
                         "(slow for 8K: one warp per stream)")
    ap.add_argument("--inflate-mode", type=int, default=0)
    ap.add_argument("--mode", default="decode", choices=["decode", "encode", "inflate"],
                    help="inflate: BASELINE.json configs[4], standalone gzip streams of --sweep-mb sizes (device-resident)")
    ap.add_argument("--sweep-mb", default="1,16,256,1024", help="--mode inflate: uncompressed stream sizes in MiB")
    ap.add_argument("--encode-level", type=int, default=9)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-batch", type=int, default=0, help="images per GPU in the host-buffer leg (0 = auto: whole batch if <= 110 GB pinned)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--e2e-gib", type=int, default=0, help="pinned host staging per rank for the end-to-end leg (GiB, upper bound; "
                    "0 = 96 on one GPU -- the whole 444-image batch -- and 24 per rank under torchrun)")
    ap.add_argument("--e2e-api", choices=["idat", "files"], default="idat",
                    help="host leg through pngb200_decode_batch (IDAT payloads) or pngb200_png_decode_batch (whole PNG files, "
                         "65544-byte IDAT chunks: chunk CRC-32 and IDAT gather on the device)")
    ap.add_argument("--e2e-sweep", default="", help="experiment: comma list of LANESxCHUNKS_PER_LANE to time the host leg with")
    ap.add_argument("--cpu-images", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one decoded (rank 0's batch) to DIR/*.npy: "
                         "per-image status, checksum and produced bytes, and a seeded sample of the pixel bytes")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.mode != "decode"):
        ap.error("--dump-outputs writes the outputs of the GPU decode path (--impl ours --mode decode)")
    return args


DUMP_SAMPLES = 1 << 22  # pixel bytes kept by --dump-outputs: 16 MiB of float32 values + 32 MiB of float64 offsets


def dump_outputs(out_dir, d_pixels, descs, B):
    """What a caller of pngb200_decode_batch receives, as float arrays: the per-image result words in full and
    the decoded pixel bytes at DUMP_SAMPLES offsets drawn from a fixed seed (the same ones for the same
    workload and batch, so that two builds can be compared output for output)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = d_pixels.numel()
    if total <= DUMP_SAMPLES:
        index = np.arange(total, dtype=np.int64)
    else:
        index = np.unique(np.random.default_rng(0).integers(0, total, DUMP_SAMPLES, dtype=np.int64))
    sample = d_pixels.view(-1)[torch.from_numpy(index).to(d_pixels.device)]
    arrays = {"status": [descs[i].status for i in range(B)], "checksum": [descs[i].checksum for i in range(B)],
              "produced": [descs[i].produced for i in range(B)], "pixels_sample": sample.float().cpu().numpy(),
              "pixels_sample_offset": index}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"),
                np.asarray(a, dtype=np.float32 if name == "pixels_sample" else np.float64))


# ------------------------------------------------------------------ corpus
def make_corpus(args, pkg, ctx):
    """U unique images -> (pixels bytes, filtered adler, zlib stream).  Filtering uses OUR
    filter-select kernel when a context exists (the oracle is only the cpu_baseline / checker)."""
    import corpus
    w, h, sixteen, _, _ = WORKLOADS[args.workload]
    bpp = 8 if sixteen else 4
    from concurrent.futures import ThreadPoolExecutor

    def synth(i):
        img = corpus.make(args.kind, w, h, i, sixteen) if args.kind == "photo" else corpus.make(args.kind, w, h, i)
        return np.ascontiguousarray(img).tobytes()

    def finish(storage, filtered):
        comp = zlib.compress(filtered, args.level) if args.encoder == "zlib" or ctx is None else None
        return dict(pixels=storage, adler=zlib.adler32(filtered), idat=comp, filtered_len=len(filtered),
                    filtered=filtered if comp is None else None)

    workers = max(1, min(args.unique, (os.cpu_count() or 4) // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))))
    with ThreadPoolExecutor(max_workers=workers) as ex:  # numpy and zlib release the GIL
        storages = list(ex.map(synth, range(args.unique)))
        if ctx is not None:
            filtered = [pkg.filter_batch(ctx, [dict(pixels=st, width=w, height=h, volume=8 * bpp,
                                                    depth=16 if sixteen else 8)])[0] for st in storages]
        else:
            from oracle import oracle
            filtered = list(ex.map(lambda st: oracle.png_filter(st, w, h, 8 * bpp, 16 if sixteen else 8), storages))
        out = list(ex.map(finish, storages, filtered))
    if ctx is not None and args.encoder == "ref":
        got = pkg.deflate_batch(ctx, [it["filtered"] for it in out], args.encode_level)
        for it, (st, comp) in zip(out, got):
            assert st == 0
            it["idat"], it["filtered"] = comp, None
    return out


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.stop, self.thread = index, [], threading.Event(), None

    def _run(self):
        while not self.stop.is_set():
            try:
                r = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.rows.append([x.strip() for x in r.stdout.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        self.thread.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


# ------------------------------------------------------------------ cpu (oracle) leg
def cpu_decode_rate(corpus_items, w, h, bpp, depth, nimages: int, threads: int):
    """MPixels/s of the CPU restatement of the reference on `nimages` decodes over `threads`
    host threads (ctypes releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import oracle
    oracle.lib()
    jobs = [corpus_items[i % len(corpus_items)] for i in range(nimages)]
    import numpy as np
    L = oracle.lib()
    local = threading.local()  # one output buffer per worker thread, allocated outside the C call

    def one(item):
        if getattr(local, "out", None) is None:
            local.out = np.empty(w * h * bpp, dtype=np.uint8)
        res = oracle.InflateResult()
        # straight into the C restatement: no Python-side copies of the 100+ MB buffers under the GIL
        st = L.orc_png_decode(oracle.ZLIB, item["idat"], len(item["idat"]), w, h, 8 * bpp, depth, 0,
                              local.out.ctypes.data, C.byref(res))
        assert st == 0 and res.checksum == item["adler"]
        return w * h * bpp

    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(one, jobs))
    dt = time.perf_counter() - t0
    return nimages * w * h / dt / 1e6, dt


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def main():
    args = parse_args()
    quiet_stdout()
    w, h, sixteen, dbatch, dunique = WORKLOADS[args.workload]
    args.batch = args.batch or dbatch
    args.unique = min(args.unique or dunique, args.batch)
    bpp, depth = (8, 16) if sixteen else (4, 8)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    enc = f"zlib level {args.level}" if args.encoder == "zlib" else f"reference-exact encoder level {args.encode_level}"
    config = {"workload": f"{args.batch}x {w}x{h} RGBA{depth} per GPU ({args.kind}, {enc}, "
                          f"reference filter rule; {args.unique} distinct images)",
              "images_per_gpu": args.batch, "l2": "inputs larger than L2 (no flush needed)"}

    # ---------------- reference arm: the CPU restatement on the host cores ----------------
    if args.impl == "reference":
        if rank != 0:
            return
        items = make_corpus(args, None, None)
        threads = os.cpu_count() or 1
        # one image per host thread and step (every core busy); 8K images are capped at 64 per step so that a
        # step stays under ~10 s on the box (measured r01: 128 threads 269 MPixels/s, 16 threads 199)
        per_step = args.cpu_images or max(min(threads, 64) if w * h > 4_000_000 else threads, 1)
        threads = min(threads, per_step)
        for _ in range(max(args.warmup, 0) and 1):
            cpu_decode_rate(items, w, h, bpp, depth, min(per_step, threads), threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_decode_rate(items, w, h, bpp, depth, per_step, threads)
        dt = time.perf_counter() - t0
        v = args.steps * per_step * w * h / dt / 1e6
        line = {"impl": "reference", "metric": "MPixels/s decode (inflate+unfilter)", "value": v, "unit": "MPixels/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": v, "unit": "MPixels/s", "cores": threads, "kind": "port",
                                 "sample": f"{per_step} images per step, {threads} host threads, C restatement "
                                           "of the Swift reference (no Swift toolchain in the image)"},
                "e2e": {"value": v, "unit": "MPixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(json.dumps(line))
        return

    if args.mode == "encode":
        return main_encode(args, w, h, bpp, depth, rank, local_rank, world, config)
    if args.mode == "inflate":
        return main_inflate(args, rank, local_rank, world)

    # ---------------- our arm ----------------
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = importlib.import_module("swift-png_b200")
    ctx = pkg.Context(local_rank)
    ctx.set_inflate_mode(args.inflate_mode)
    stream = torch.cuda.ExternalStream(ctx.stream, device=local_rank)
    items = make_corpus(args, pkg, ctx)
    B = args.batch
    npix = w * h
    storage_bytes = npix * bpp

    # device-resident inputs -- one private copy of its stream per job, so the compressed bytes of a
    # step (several GB) cannot sit in the 126 MB L2 -- and outputs
    d_unique = [torch.frombuffer(bytearray(it["idat"]), dtype=torch.uint8).cuda() for it in items]
    d_idat = [d_unique[i % len(items)].clone() for i in range(B)]
    del d_unique
    d_pixels = torch.empty((B, storage_bytes), dtype=torch.uint8, device="cuda")
    descs = (pkg.ImageDesc * B)()
    for i in range(B):
        u = i
        descs[i].idat = d_idat[u].data_ptr()
        descs[i].idat_len = d_idat[u].numel()
        descs[i].pixels = d_pixels[i].data_ptr()
        descs[i].pixels_cap = storage_bytes
        descs[i].width, descs[i].height = w, h
        descs[i].volume, descs[i].depth = 8 * bpp, depth
        descs[i].interlaced, descs[i].format = 0, 0
    L = ctx._lib

    shard = importlib.import_module("swift-png_b200.shard")
    gather_device = torch.device("cuda", local_rank)
    comp_sizes = [d_idat[i % B].numel() for i in range(B)] * world  # every rank holds B jobs of the same sizes

    def decode_my_shard(_indices):
        ctx.check(L.pngb200_decode_batch_enqueue(ctx.handle, descs, B, pkg.MEM_DEVICE))
        ctx.check(L.pngb200_decode_batch_finish(ctx.handle, descs, B))  # synchronises the library's stream
        return [(descs[i].status, descs[i].checksum, descs[i].produced) for i in range(B)]

    def step_device():
        if world == 1:
            decode_my_shard(None)
            return
        # the only collective of the path (swift-png_b200/shard.py): every rank learns the whole batch's
        # per-image (status, adler32, produced) words; decoded pixels stay sharded on the GPU that produced
        # them.  The gather is issued after this rank's kernels have finished (finish() synchronised) and
        # its result is consumed on the host before the next step starts, so no NCCL kernel is co-resident
        # with the next step's inflate kernel
        rows = shard.run_sharded(comp_sizes, decode_my_shard, device=gather_device, equal_shards=B)
        assert len(rows) == world * B and all(r[0] == 0 for r in rows), "a rank reported a failed image"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step_device()
    # bit-exactness in the same run: round trip == original pixels, Adler-32 == zlib's
    torch.cuda.synchronize()
    for u, it in enumerate(items):
        ref = torch.frombuffer(bytearray(it["pixels"]), dtype=torch.uint8).cuda()
        for i in range(u, B, len(items)):
            if os.environ.get("PNGB200_BENCH_NOVERIFY"):   # timing experiments with deliberately broken kernels only
                continue
            assert descs[i].status == 0, (i, descs[i].status)
            assert descs[i].checksum == it["adler"], i
            assert torch.equal(d_pixels[i], ref), f"pixel mismatch in image {i}"
        del ref
    launches0 = ctx.launches
    stage = np.zeros(3)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local_rank) as clocks:
        ev0.record(stream)
        for _ in range(args.steps):
            step_device()
            stage += np.array(ctx.stage_ms())
        ev1.record(stream)
        barrier()
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_pixels, descs, B)
    stats = ctx.inflate_counters(B)
    engine_used = ctx.last_inflate_engine()
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * npix * args.steps / (ms_max / 1e3) / 1e6
    stage /= args.steps

    # ---------------- the 8-images-per-GPU row (BASELINE configs[3]'s per-GPU shape, SURVEY 8d "metric row"):
    # fewer streams than CTA slots, so every stream is cut into segments (csrc/inflate_segments.cuh) ----------------
    small = None
    if B >= 8:
        SB = 8
        for _ in range(2):
            ctx.check(L.pngb200_decode_batch_enqueue(ctx.handle, descs, SB, pkg.MEM_DEVICE))
            ctx.check(L.pngb200_decode_batch_finish(ctx.handle, descs, SB))
        seg = ctx.segment_stats()
        assert os.environ.get("PNGB200_BENCH_NOVERIFY") or all(descs[i].status == 0 and descs[i].checksum == items[i % len(items)]["adler"] for i in range(SB))
        assert os.environ.get("PNGB200_BENCH_NOVERIFY") or torch.equal(d_pixels[SB - 1], torch.frombuffer(bytearray(items[(SB - 1) % len(items)]["pixels"]), dtype=torch.uint8).cuda())
        torch.cuda.synchronize()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        for _ in range(3):
            ctx.check(L.pngb200_decode_batch_enqueue(ctx.handle, descs, SB, pkg.MEM_DEVICE))
            ctx.check(L.pngb200_decode_batch_finish(ctx.handle, descs, SB))
        s1.record(stream)
        torch.cuda.synchronize()
        sms = s0.elapsed_time(s1) / 3
        small = {"images_per_gpu": SB, "value": SB * npix / (sms / 1e3) / 1e6, "unit": "MPixels/s (this GPU)", "ms_per_step": sms,
                 "segments": seg["segments"], "segment_fallbacks": seg["fallbacks"], "stage_ms": dict(zip(("inflate", "checksum", "unfilter"), ctx.stage_ms())),
                 "counters": ctx.inflate_counters(SB)}

    # ---------------- e2e: same call, HOST (pinned) buffers, copies inside the timed region ----------------
    e2e = None
    if not args.no_e2e:
        import psutil
        per_image = storage_bytes + max(len(it["idat"]) for it in items)
        # Pinned host staging per rank: min(96 GiB alone / 24 GiB per rank under torchrun, 30 % of the free host memory / ranks), decided ONCE
        # on rank 0 and broadcast, so that every rank times the same sub-batch and 8 ranks cannot pin the box
        # to death (r01 lost its 8-GPU run to 94 GB of pinned memory per rank)
        gib = args.e2e_gib or (96 if world == 1 else 24)
        budget = min(gib << 30, int(0.3 * psutil.virtual_memory().available / max(world, 1)))
        EB = max(8, min(B, args.e2e_batch or B, budget // per_image))
        if world > 1:
            eb = torch.tensor([EB], dtype=torch.int64, device="cuda")
            dist.broadcast(eb, 0)
            EB = int(eb.item())
        full_B, B = B, EB
        if args.e2e_api == "files":
            import struct
            import zlib

            def chunk(t, body):
                return struct.pack(">I", len(body)) + t + body + struct.pack(">I", zlib.crc32(t + body))

            for it in items:  # the file the reference's encoder would frame around this IDAT payload
                z = it["idat"]
                it["file"] = (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, 6, 0, 0, 0)) +
                              b"".join(chunk(b"IDAT", z[o:o + 65544]) for o in range(0, len(z), 65544)) + chunk(b"IEND", b""))
        src_key = "file" if args.e2e_api == "files" else "idat"
        comp_total = sum(len(items[i % len(items)][src_key]) for i in range(B))
        h_in = torch.empty(comp_total, dtype=torch.uint8, pin_memory=True)   # cudaHostAlloc directly: no pageable twin
        h_out = torch.empty((B, storage_bytes), dtype=torch.uint8, pin_memory=True)
        hdescs = (pkg.PngDesc * B)() if args.e2e_api == "files" else (pkg.ImageDesc * B)()
        at = 0
        for i in range(B):
            it = items[i % len(items)]
            n = len(it[src_key])
            h_in[at:at + n] = torch.frombuffer(bytearray(it[src_key]), dtype=torch.uint8)
            hdescs[i].pixels = h_out[i].data_ptr()
            hdescs[i].pixels_cap = storage_bytes
            if args.e2e_api == "files":
                hdescs[i].file, hdescs[i].file_len = h_in.data_ptr() + at, n
            else:
                hdescs[i].idat = h_in.data_ptr() + at
                hdescs[i].idat_len = n
                hdescs[i].width, hdescs[i].height = w, h
                hdescs[i].volume, hdescs[i].depth = 8 * bpp, depth
            at += n
        del d_pixels, d_idat, descs
        torch.cuda.empty_cache()
        ctx.trim()  # the device-resident leg's arenas would otherwise sit beside the lanes'

        def step_host():
            if args.e2e_api == "files":
                ctx.check(L.pngb200_png_decode_batch(ctx.handle, hdescs, B, pkg.MEM_HOST))
                assert all(hdescs[i].status == 0 for i in range(0, B, max(1, B // 8)))
            else:
                ctx.check(L.pngb200_decode_batch(ctx.handle, hdescs, B, pkg.MEM_HOST))

        for _ in range(2):
            step_host()
        assert bytes(h_out[B - 1].numpy().tobytes()) == items[(B - 1) % len(items)]["pixels"]
        barrier()
        t0 = time.perf_counter()
        esteps = max(1, min(args.steps, 3))
        for _ in range(esteps):
            step_host()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * B * npix * esteps / float(dt.item()) / 1e6, "unit": "MPixels/s",
               "h2d_bytes_per_step": comp_total, "d2h_bytes_per_step": B * storage_bytes, "steps": esteps,
               "pcie_ceiling": {"value": 44.7e9 / (storage_bytes / npix) / 1e6 * world, "unit": "MPixels/s",
                                "note": "D2H of the decoded pixels at the 44.7 GB/s this box moves each way when both "
                                        "directions run (profiles/r01_pcie_bandwidth.json)"},
               "images_per_gpu": B, "api": "pngb200_png_decode_batch" if args.e2e_api == "files" else "pngb200_decode_batch",
               "note": ("whole PNG files (65544-byte IDAT chunks) in pinned HOST memory: chunk walk on the host, "
                        "chunk CRC-32, IDAT gather, inflate and unfilter on the device; "
                        if args.e2e_api == "files" else "pngb200_decode_batch with pinned HOST buffers: ") +
                       "H2D of the compressed bytes and D2H of the decoded pixels are inside the timed region "
                       "(host wall clock, max over ranks)"}
        if args.e2e_sweep:
            sweep = {}
            for cfg in args.e2e_sweep.split(","):
                ln, ck = cfg.split("x")
                os.environ["PNGB200_LANES"], os.environ["PNGB200_CHUNKS_PER_LANE"] = ln, ck
                try:
                    ctx.trim()
                    step_host()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(2):
                        step_host()
                    sweep[cfg] = B * npix * 2 / (time.perf_counter() - t0) / 1e6
                except Exception as exc:  # e.g. a chunking that does not fit the device
                    sweep[cfg] = "failed: %s" % (str(exc)[:80],)
            e2e["sweep"] = sweep
            os.environ.pop("PNGB200_LANES"), os.environ.pop("PNGB200_CHUNKS_PER_LANE")
        B = full_B

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (inflate), measured live ----------------
    peak, peak_src = peaks()
    comp_step = sum(len(items[i % len(items)]["idat"]) for i in range(B))
    alg_bytes = comp_step + B * storage_bytes  # SURVEY 8(d): C + P per image x images per launch
    dominant = int(np.argmax(stage))
    inflate_kernel = engine_used or ("inflate_wave_kernel" if B <= 296 else "inflate_parallel_kernel")  # as reported by run_inflate
    names = [inflate_kernel, "checksum kernels", "unfilter_wave_kernel"]
    achieved = alg_bytes / (stage[0] / 1e3) / 1e9
    traffic, issue = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        for entry in json.load(open(tpath)).get(args.workload) or []:
            if entry.get("batch") == B and entry.get("kernel") == inflate_kernel and args.encoder == "zlib" and args.kind == "photo":
                traffic = entry["bytes_per_launch"]  # measured once under ncu for exactly this launch shape
                if entry.get("warp_instructions_per_launch"):
                    # issue roofline beside the HBM one: warp instructions of the launch (ncu) over what the
                    # SMs' 4 schedulers can issue in the measured time at the sampled SM clock
                    clk = (clocks.summary().get("sm_mhz") or 1965.0) * 1e6
                    issue = {"warp_instructions_per_launch": entry["warp_instructions_per_launch"],
                             "per_output_byte": entry["warp_instructions_per_launch"] / (B * pkg.filtered_size(w, h, 8 * bpp)),
                             "frac": entry["warp_instructions_per_launch"] / (148 * 4 * clk * stage[0] / 1e3)}
    roofline = {"bound": "hbm", "kernel": names[0], "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes,
                "stage_ms": {"inflate": stage[0], "checksum": stage[1], "unfilter": stage[2]},
                "dominant_stage": names[dominant], "issue_roofline": issue,
                "whole_step_frac": alg_bytes / (ms_max / args.steps / 1e3) / 1e9 / peak}

    cpu = None
    if not args.no_cpu and world == 1:  # the host-core baseline is reported at N = 1 only
        threads = os.cpu_count() or 1
        n_cpu = args.cpu_images or (threads if npix > 4_000_000 else 4 * threads)
        v, dt = cpu_decode_rate(items, w, h, bpp, depth, n_cpu, threads)
        v1, dt1 = cpu_decode_rate(items, w, h, bpp, depth, 2 if npix > 4_000_000 else 8, 1)
        cpu = {"value": v, "unit": "MPixels/s", "cores": threads, "kind": "port", "one_thread": v1,
               "sample": f"{n_cpu} images of the same workload over {threads} host threads in {dt:.1f}s "
                         f"(one thread alone: {v1:.1f} MPixels/s); C restatement of the Swift reference (oracle/, "
                         "thread-local scratch), no Swift toolchain in the image"}

    line = {"metric": "MPixels/s decode (inflate+unfilter)", "value": value, "unit": "MPixels/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config, "clocks": clocks.summary(), "gpu_launches": int(launches),
            "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu, "bit_exact": True, "small_batch": small,
            "inflate_stats_per_step": stats}
    emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main_inflate(args, rank, local_rank, world):
    """BASELINE.json configs[4]: standalone LZ77 / Gzip.Inflator throughput on gzip streams of S0 filtered
    bytes (SURVEY section 8d config 5), device-resident, one JSON line with two rows per stream size: ONE stream
    (cut into segments, one CTA each: csrc/inflate_segments.cuh) and min(296, ~6 GiB / size) independent streams."""
    import zlib

    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import corpus
    torch.cuda.set_device(local_rank)
    pkg = importlib.import_module("swift-png_b200")
    ctx = pkg.Context(local_rank)
    L = ctx._lib
    stream = torch.cuda.ExternalStream(ctx.stream, device=local_rank)
    base = b"".join(corpus.zlib_png_stream(corpus.make("photo", 2048, 1024, 0x5EED + k), 4, 6)[0] for k in range(2))
    rows = []
    for mb in [int(x) for x in args.sweep_mb.split(",")]:
        n = mb << 20
        plain = (base * (n // len(base) + 1))[:n]
        co = zlib.compressobj(6, zlib.DEFLATED, 31)  # gzip wrapper
        z = co.compress(plain) + co.flush()
        crc = zlib.crc32(plain)
        d_src = torch.frombuffer(bytearray(z), dtype=torch.uint8).cuda()
        for count in sorted({1, max(1, min(296, (6 << 30) // n))}):
            d_in = [d_src.clone() for _ in range(count)]
            d_out = torch.empty((count, n), dtype=torch.uint8, device="cuda")
            descs = (pkg.StreamDesc * count)()
            for i in range(count):
                descs[i].src, descs[i].src_len = d_in[i].data_ptr(), len(z)
                descs[i].dst, descs[i].dst_cap = d_out[i].data_ptr(), n
                descs[i].format = pkg.FORMAT_GZIP
            for _ in range(2):
                ctx.check(L.pngb200_inflate_batch(ctx.handle, descs, count, pkg.MEM_DEVICE))
            seg = ctx.segment_stats()
            assert all(descs[i].status == 0 and descs[i].produced == n for i in range(count))
            assert descs[0].checksum == crc and bytes(d_out[count - 1].cpu().numpy().tobytes()) == plain
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            steps = max(1, args.steps)
            for _ in range(steps):
                ctx.check(L.pngb200_inflate_batch(ctx.handle, descs, count, pkg.MEM_DEVICE))
            e1.record(stream)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            rows.append({"stream_mib": mb, "streams": count, "compressed_bytes": len(z), "ms_per_batch": ms,
                         "out_GBps": count * n / ms / 1e6, "c_plus_u_GBps": count * (n + len(z)) / ms / 1e6,
                         "per_stream_MBps": n / ms / 1e3, "segments": seg["segments"], "segment_fallbacks": seg["fallbacks"]})
            del d_in, d_out
            torch.cuda.empty_cache()
            ctx.trim()
        del d_src
    if rank == 0:
        best = max(r["c_plus_u_GBps"] for r in rows)
        emit(json.dumps({"metric": "GB/s standalone gzip inflate (C+U)", "value": best, "unit": "GB/s", "n_gpus": world,
                          "steps": args.steps, "warmup": 2, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "u8", "data": "synthetic",
                          "config": {"workload": "gzip streams of S0 filtered bytes, zlib level 6 (BASELINE configs[4])"},
                          "sweep": rows, "bit_exact": True}))


def main_encode(args, w, h, bpp, depth, rank, local_rank, world, config):
    """BASELINE.json config 3: batch encode (filter select + deflate level 9), MPixels/s."""
    enc = f"zlib level {args.level}" if args.encoder == "zlib" else f"reference-exact encoder level {args.encode_level}"
    import torch
    import torch.distributed as dist
    import corpus
    npix, storage_bytes = w * h, w * h * bpp
    config = dict(config, workload=config["workload"].replace(enc, "encode level %d" % args.encode_level))
    imgs = [np.ascontiguousarray(corpus.make(args.kind, w, h, i, depth == 16) if args.kind == "photo"
                                 else corpus.make(args.kind, w, h, i)).tobytes() for i in range(args.unique)]
    if args.impl == "reference":
        if rank != 0:
            return
        from concurrent.futures import ThreadPoolExecutor
        from oracle import oracle
        oracle.lib()
        threads = os.cpu_count() or 1
        per_step = args.cpu_images or min(threads, 32)

        def one(i):
            f = oracle.png_filter(imgs[i % len(imgs)], w, h, 8 * bpp, depth)
            return len(oracle.deflate(f, args.encode_level))

        t0 = time.perf_counter()
        for _ in range(args.steps):
            with ThreadPoolExecutor(max_workers=threads) as ex:
                list(ex.map(one, range(per_step)))
        dt = time.perf_counter() - t0
        v = args.steps * per_step * npix / dt / 1e6
        emit(json.dumps({"impl": "reference", "metric": "MPixels/s encode (filter+deflate)", "value": v,
                          "unit": "MPixels/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": v, "unit": "MPixels/s", "cores": threads, "kind": "port",
                                           "sample": f"{per_step} images per step over {threads} host threads"},
                          "e2e": {"value": v, "unit": "MPixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = importlib.import_module("swift-png_b200")
    ctx = pkg.Context(local_rank)
    L, B = ctx._lib, args.batch
    stream = torch.cuda.ExternalStream(ctx.stream, device=local_rank)
    cap = L.pngb200_deflate_bound(pkg.filtered_size(w, h, 8 * bpp))
    d_px = [torch.frombuffer(bytearray(imgs[i % len(imgs)]), dtype=torch.uint8).cuda() for i in range(B)]
    d_out = torch.empty((B, cap), dtype=torch.uint8, device="cuda")
    descs = (pkg.EncodeDesc * B)()
    for i in range(B):
        descs[i].pixels, descs[i].pixels_len = d_px[i].data_ptr(), storage_bytes
        descs[i].idat, descs[i].idat_cap = d_out[i].data_ptr(), cap
        descs[i].width, descs[i].height = w, h
        descs[i].volume, descs[i].depth, descs[i].level = 8 * bpp, depth, args.encode_level

    def step():
        ctx.check(L.pngb200_encode_batch(ctx.handle, descs, B, pkg.MEM_DEVICE))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3) if B * npix < 3e8 else 1):
        step()
    assert all(descs[i].status == 0 for i in range(B))
    launches0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    with ClockSampler(local_rank) as clocks:
        ev0.record(stream)
        for _ in range(args.steps):
            step()
        ev1.record(stream)
        barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    if rank != 0:
        return
    comp = sum(descs[i].produced for i in range(B))
    # bit-exactness in the same run: image 0's IDAT payload == the CPU restatement's, and it inflates
    from oracle import oracle
    mine = bytes(d_out[0, : descs[0].produced].cpu().numpy().tobytes())
    t0 = time.perf_counter()
    ref = oracle.deflate(oracle.png_filter(imgs[0], w, h, 8 * bpp, depth), args.encode_level)
    cpu_dt = time.perf_counter() - t0
    assert mine == ref, "encode output differs from the oracle"
    peak, peak_src = peaks()
    alg = B * storage_bytes + comp
    value = world * B * npix * args.steps / (ms / 1e3) / 1e6
    line = {"metric": "MPixels/s encode (filter+deflate)", "value": value, "unit": "MPixels/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
            "clocks": clocks.summary(), "gpu_launches": int(ctx.launches - launches0), "e2e": None,
            "roofline": {"bound": "hbm", "kernel": "deflate_kernel", "achieved": alg / (ms / args.steps / 1e3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": alg / (ms / args.steps / 1e3) / 1e9 / peak,
                         "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg},
            "cpu_baseline": {"value": npix / cpu_dt / 1e6, "unit": "MPixels/s", "cores": 1, "kind": "port",
                             "sample": f"1 image of the same workload on 1 host thread in {cpu_dt:.1f}s (oracle/)"},
            "bit_exact": True, "compression_ratio": B * storage_bytes / comp}
    emit(json.dumps(line))


if __name__ == "__main__":
    main()
