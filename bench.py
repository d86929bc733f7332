#!/usr/bin/env python
"""bench.py -- encode+decode MPix/s of the jpezy hot path on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4] [--impl reference] [--dump-outputs DIR]

A step = one pass of the hot path over one batch of synthetic input per GPU:
  c2 (default, BASELINE.json configs[1]): one 3840x2160 RGB image, encode then decode
  c3: a batch of 1920x1080 frames per GPU (configs[2] sharded by image; --batch frames per GPU)
  c4: one 8192x8192 image in --gray mode (configs[3])
`value` is device-timed (CUDA events, inputs resident in HBM, max over ranks); `e2e` is the same metric
through the host-buffer C-ABI calls (jpezyb200_encode / jpezyb200_decode) with pinned host buffers and the
H2D/D2H copies inside the timed region.  L2: inputs/outputs rotate through a ring of distinct frames whose
footprint exceeds the 126 MB L2 (see config.l2).

--dump-outputs DIR writes what the last timed step returned to its caller (rank 0, by-image workloads) as float32 / float64
.npy files, so that two builds can be compared output for output on identical seeded inputs:
  segments.npy       the entropy-coded segments of the step's images, concatenated (a seeded sample when large)
  segment_bytes.npy  the length of each image's segment
  decoded.npy        the decoded planes, [3, batch, plane bytes] flattened (a seeded sample when large)
"""
import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

WORKLOADS = {
    "c2": dict(W=3840, H=2160, batch=1, gray=False, name="C2: single 3840x2160 RGB image, encode+decode round trip"),
    "c3": dict(W=1920, H=1080, batch=64, gray=False, name="C3: batch of 1920x1080 RGB frames sharded by image, encode+decode"),
    "c4": dict(W=8192, H=8192, batch=1, gray=True, name="C4: single 8192x8192 --gray image, encode+decode"),
    "c1": dict(W=512, H=512, batch=1, gray=False, name="C1: single 512x512 RGB image, encode+decode"),
    "c5": dict(W=32768, H=32768, batch=1, gray=False, name="C5: single 32768x32768 RGB image, encode split by MCU rows across the GPUs"),
}
FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON result: everything else libraries print there (NCCL's version banner, ...)
    is sent to stderr -- file descriptor 1 is pointed at stderr, the real one is kept for emit()"""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """samples SM clock / throttle reasons of one GPU every 20 ms through NVML while the bench runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag, self.ok = index, [], set(), None, False, False
        self.mark = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if self.mark is not None:
                    self.samples.append(mhz)
                    for k, bit in names.items():
                        if mask & bit:
                            self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def cpu_arm():
    """The reference's CPU implementation of the path: oracle/_ref (the reference's own sources compiled against
    oracle/shim, SURVEY.md 8c / DESIGN.md) when it was built, else the oracle port.  -> (timer, kind)
    timer(r, g, b, W, H, gray, reps, ninstances) -> (wall s, encode s, decode s)"""
    import oracle as orc
    if orc.ref_dir() is not None:
        ref = orc.Reference()
        return ref.time_roundtrip, "reference"
    orc.build()
    o = orc.Oracle("shipped")      # the reference's Release flags (compiler_settings.cmake:4)
    return o.time_roundtrip, "port"


def run_reference(args, wl):
    """--impl reference: the reference's own encoder::encode() + decoder::decode() on all host cores (one instance per
    core, the reference is single threaded), each step a bounded sample of the workload image."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import jpezy_b200 as J
    timer, kind = cpu_arm()
    cores = os.cpu_count() or 1
    W, H = wl["W"], wl["H"]
    # bounded sample: a band of MCU rows of the workload image, sized for ~120 s total at ~2.7 MPix/s/core round trip
    budget_px = 120.0 / max(1, args.steps + args.warmup) * 2.7e6
    rows = int(min(H, max(16, (budget_px // W) // 16 * 16)))
    r, g, b = J.synth.image(0, W, rows, frame=0)
    for _ in range(args.warmup):
        timer(r, g, b, W, rows, wl["gray"], 1, cores)
    dt = te = td = 0.0
    for _ in range(args.steps):
        w, e, d = timer(r, g, b, W, rows, wl["gray"], 1, cores)
        dt += w
        te += e
        td += d
    px = float(W) * rows * cores * args.steps
    val = px / dt / 1e6
    sample = "%dx%d band (%d of %d rows) of the workload image per instance, %d concurrent single-threaded instances, " \
             "encode()+decode() per step, PNM I/O excluded" % (W, rows, rows, H, cores)
    line = {"impl": "reference", "metric": "encode+decode MPix/s", "value": val, "unit": "MPix/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["name"], "width": W, "height": H, "batch_per_gpu": wl["batch"], "gray": wl["gray"],
                       "family": "S-photo"},
            "cpu_baseline": {"value": val, "unit": "MPix/s", "cores": cores, "kind": kind, "sample": sample,
                             "encode_MPix_s_per_core": float(W) * rows * args.steps / te / 1e6 if te else None,
                             "decode_MPix_s_per_core": float(W) * rows * args.steps / td / 1e6 if td else None},
            "e2e": {"value": val, "unit": "MPix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def run_sharded(args, wl):
    """C5: ONE giant image, encode only, sharded by MCU rows over the ranks (strong scaling): transform local rows,
    all-gather DC predictors / bit counts / byte counts (NCCL), stitched stream written into rank 0's buffer over NVLink."""
    import numpy as np
    import torch
    import jpezy_b200 as J
    from jpezy_b200 import capi, shard
    args.steps = args.steps or 20
    args.warmup = max(args.warmup if args.warmup is not None else 3, 3)
    rank, local_rank, world = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1")))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    ctx = J.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    W, H, gray = args.width or wl["W"], args.height or wl["H"], wl["gray"]
    VU = (H + 15) // 16
    row0, nrows = shard.partition_mcu_rows(VU, world)[rank]
    y0, ny = shard.pixel_rows(H, row0, nrows)
    sampler = ClockSampler(local_rank)
    sampler.start()
    planes = torch.empty((3, ny, W), dtype=torch.uint8, device="cuda")       # > L2 on every rank for the named shape
    ctx.synth_rows_dev(planes[0], planes[1], planes[2], W, y0, ny, frame=0, family=args.family, stream=sp)
    grp = shard.DistGroup(dist, torch.device("cuda", local_rank))
    dst_cap = max(W * H // 2, 1 << 20)
    enc = shard.ShardedEncoder(ctx, grp, dst_cap)

    def step():
        enc.encode(planes[0], planes[1], planes[2], W, H, row0, nrows, y0, gray, stream=sp)

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler.mark = True
    l0 = ctx.stat(capi.STAT_KERNEL_LAUNCHES)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.stat(capi.STAT_KERNEL_LAUNCHES) - l0
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # the dominant kernel: forward transform of the local rows
    def fwd():
        ctx.shard_encode_a(planes[0], planes[1], planes[2], W, H, row0, nrows, y0, gray, enc.last_dc, stream=sp)
    for _ in range(3):
        fwd()
    torch.cuda.synchronize()
    a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(10):
        fwd()
    b2.record(stream)
    torch.cuda.synchronize()
    t_fwd = a.elapsed_time(b2) / 10
    sampler.mark = None
    seg, bits = enc.result()
    sampler.stop_flag = True
    peak, peak_src = measured_peak()
    alg = 6.0 * W * 16 * nrows
    if rank == 0:
        value = float(W) * H * args.steps / (ms * 1e-3) / 1e6
        line = {"metric": "encode MPix/s", "value": value, "unit": "MPix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": wl["name"], "width": W, "height": H, "gray": gray, "family": "S-photo" if args.family == 0 else "S-noise",
                           "l2": "inputs larger than L2 (%.0f MB of planes per rank)" % (3.0 * ny * W / 1e6),
                           "sharding": "MCU rows, %d per rank; 3 all-gathers (12 B, 16 B, 8 B per rank) + P2P stores of the stuffed segment into rank 0" % nrows},
                "clocks": sampler.summary(), "gpu_launches": int(launches), "e2e": None,
                "roofline": {"bound": "hbm", "kernel": "k_fwd_transform", "achieved": alg / (t_fwd * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": alg / (t_fwd * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg, "ms_per_launch": t_fwd},
                "cpu_baseline": None,
                "stages": {"stream_bytes": len(seg), "bits_per_rank": bits, "fwd_transform_ms_rank0": t_fwd}}
        emit(line)
    enc.close()
    dist.destroy_process_group()
    ctx.close()


def run_sharded_gray(args, wl):
    """C4 on N GPUs, --shard: ONE 8192x8192 --gray image, encode sharded by MCU rows (collectives + P2P stitch) then decode with
    the entropy stage replicated on every rank and the transform stage sharded by MCU rows (P2P stores into rank 0's planes)."""
    import torch
    import torch.distributed as dist
    import jpezy_b200 as J
    from jpezy_b200 import capi, shard
    args.steps = args.steps or 20
    args.warmup = max(args.warmup if args.warmup is not None else 3, 3)
    rank, local_rank, world = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1")))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = J.Context(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    W, H, gray = args.width or wl["W"], args.height or wl["H"], True
    row0, nrows = shard.partition_mcu_rows((H + 15) // 16, world)[rank]
    y0, ny = shard.pixel_rows(H, row0, nrows)
    sampler = ClockSampler(local_rank)
    sampler.start()
    planes = torch.empty((3, ny, W), dtype=torch.uint8, device="cuda")
    ctx.synth_rows_dev(planes[0], planes[1], planes[2], W, y0, ny, frame=0, family=args.family, stream=sp)
    grp = shard.DistGroup(dist, torch.device("cuda", local_rank))
    cap = max(W * H // 2, 1 << 20)
    enc = shard.ShardedEncoder(ctx, grp, cap)
    frame = J.default_frame(W, H)
    dec = shard.ShardedDecoder(ctx, grp, frame, cap)
    enc.encode(planes[0], planes[1], planes[2], W, H, row0, nrows, y0, gray, stream=sp)
    seg, _ = enc.result()
    nbytes = torch.zeros(1, dtype=torch.int64, device="cuda")
    if rank == 0:
        nbytes[0] = len(seg)
        dec.scan[: len(seg)] = torch.frombuffer(bytearray(seg), dtype=torch.uint8).cuda()
    dist.broadcast(nbytes, src=0)
    n_scan = int(nbytes.item())

    def step():
        enc.encode(planes[0], planes[1], planes[2], W, H, row0, nrows, y0, gray, stream=sp)
        dec.decode(n_scan, gray, stream=sp)        # (the stream of the previous encode: same bytes every step)

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
    for _ in range(args.warmup):
        step()
    barrier()
    sampler.mark = True
    l0 = ctx.stat(capi.STAT_KERNEL_LAUNCHES)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.stat(capi.STAT_KERNEL_LAUNCHES) - l0
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    sampler.mark = None
    out = dec.result()
    sampler.stop_flag = True
    if rank == 0:
        ok = bool(out is not None and out[0][: W * 16].any())
        line = {"metric": "encode+decode MPix/s", "value": float(W) * H * args.steps / (ms * 1e-3) / 1e6, "unit": "MPix/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
                "config": {"workload": wl["name"] + " (one image sharded by MCU rows)", "width": W, "height": H, "gray": True,
                           "family": "S-photo" if args.family == 0 else "S-noise", "l2": "inputs larger than L2",
                           "sharding": "encode: MCU rows + 3 all-gathers + P2P stitch; decode: segment broadcast, entropy stage replicated, "
                                       "transform stage by MCU rows with P2P stores into rank 0"},
                "clocks": sampler.summary(), "gpu_launches": int(launches), "e2e": None, "roofline": None, "cpu_baseline": None,
                "stages": {"stream_bytes": n_scan, "decoded_ok": ok}}
        emit(line)
    dec.close()
    enc.close()
    dist.destroy_process_group()
    ctx.close()


def extra_configs(args, ctx, dist, rank, local_rank, world):
    """The other BASELINE.json configurations, measured in the same process right after the headline workload (a few steps
    each; device-timed like the headline, max over ranks).  Returned on rank 0 as the `configs` object of the JSON line:
      c3        batch of 1920x1080 frames, 64 per GPU, sharded by image (weak scaling, no data-path collective)
      c5        ONE 32768x32768 image, encode sharded by MCU rows (strong scaling): total, the seven phases of the sharded
                encoder (which all-gather or kernel limits it) and the SHA-256 of the stitched segment against the segment
                rank 0 encodes alone from the same pixels
      c4_shard  ONE 8192x8192 --gray image, encode + decode sharded by MCU rows; decoded planes against a single-GPU decode"""
    import hashlib
    import numpy as np
    import torch
    import jpezy_b200 as J
    from jpezy_b200 import capi, shard
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream
    peak, _ = measured_peak()
    out = {}
    own_group = False
    if dist is None:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", local_rank))
        own_group = True

    def rank_max(ms):
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sync_all():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(fn, warm, steps):
        for i in range(warm):
            fn(i)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            fn(i)
        e1.record(stream)
        sync_all()
        return rank_max(e0.elapsed_time(e1)) / steps

    # ---- C3: batch by image ----
    try:
        W, H, B = 1920, 1080, 64
        npx = W * H
        frame = J.default_frame(W, H)
        pl = J.plane_bytes(frame)
        ring = 2                                                   # 2 x (398 + 398) MB of frames: far above the 126 MB L2
        slot = npx
        d_in = torch.empty((ring, 3, B, H, W), dtype=torch.uint8, device="cuda")
        d_out = torch.zeros((ring, 3, B, pl), dtype=torch.uint8, device="cuda")
        d_scan = torch.zeros((ring, B, slot), dtype=torch.uint8, device="cuda")
        d_nb = torch.zeros((ring, B), dtype=torch.int64, device="cuda")
        d_st = torch.zeros((ring, B), dtype=torch.int32, device="cuda")
        d_coefs = torch.empty((B, capi.num_mcus(W, H), 6, 64), dtype=torch.int16, device="cuda")
        for k in range(ring):
            ctx.synth_dev(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, nimg=B, first_frame=(rank * ring + k) * B, family=args.family, stream=sp)
            ctx.encode_batch_dev(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, B, False, d_scan[k], slot, d_nb[k], None, stream=sp)
        torch.cuda.synchronize()
        h_nb = d_nb.cpu().numpy().astype(np.uint64)
        bound = min(slot, int(h_nb.max() * 1.25) + 4096)

        def step(i):
            k = i % ring
            ctx.encode_batch_dev(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, B, False, d_scan[k], slot, d_nb[k], None, stream=sp)
            ctx.decode_batch_dev2(d_scan[k], slot, d_nb[k], bound, B, frame, False, d_out[k, 0], d_out[k, 1], d_out[k, 2], pl, d_st[k], stream=sp)
        ms = timed_loop(step, 3, 10)
        assert int(d_st.abs().sum().item()) == 0
        t = {}
        t["fwd_transform_ms"] = timed_loop(lambda i: ctx.transform_fwd_dev(d_in[i % ring, 0], d_in[i % ring, 1], d_in[i % ring, 2], W, H, B, False, d_coefs, stream=sp), 2, 8)
        t["entropy_encode_ms"] = timed_loop(lambda i: ctx.entropy_encode_dev(d_coefs, W, H, B, False, d_scan[i % ring], slot, d_nb[i % ring], None, stream=sp), 2, 8)
        t["entropy_decode_ms"] = timed_loop(lambda i: ctx.entropy_decode_dev(d_scan[i % ring], slot, h_nb[i % ring], B, frame, d_coefs, d_st[i % ring], stream=sp), 2, 8)
        t["inv_transform_ms"] = timed_loop(lambda i: ctx.transform_inv_dev(d_coefs, frame, B, False, d_out[i % ring, 0], d_out[i % ring, 1], d_out[i % ring, 2], pl, stream=sp), 2, 8)
        out["c3"] = {"workload": "batch of 1920x1080 RGB frames sharded by image", "batch_per_gpu": B, "n_gpus": world, "scaling": "weak",
                     "value": world * B * npx / (ms * 1e-3) / 1e6, "unit": "MPix/s", "ms_per_step": ms, "steps": 10, "stages": t,
                     "fwd_transform_frac_of_hbm": 6.0 * B * npx / (t["fwd_transform_ms"] * 1e-3) / 1e9 / peak,
                     "inv_transform_frac_of_hbm": 6.0 * B * npx / (t["inv_transform_ms"] * 1e-3) / 1e9 / peak,
                     "bits_per_pixel": float(h_nb.mean()) * 8 / npx}
        del d_in, d_out, d_scan, d_coefs
        torch.cuda.empty_cache()
    except Exception as e:       # a configuration that cannot run here is reported, the headline line still prints
        out["c3"] = {"error": repr(e)[:300]}

    grp = shard.DistGroup(dist, torch.device("cuda", local_rank))

    # ---- C5: one giant image, encode sharded by MCU rows ----
    try:
        W = H = 32768
        VU = (H + 15) // 16
        row0, nrows = shard.partition_mcu_rows(VU, world)[rank]
        y0, ny = shard.pixel_rows(H, row0, nrows)
        planes = torch.empty((3, ny, W), dtype=torch.uint8, device="cuda")
        ctx.synth_rows_dev(planes[0], planes[1], planes[2], W, y0, ny, frame=0, family=args.family, stream=sp)
        cap = W * H // 2
        enc = shard.ShardedEncoder(ctx, grp, cap)
        ms = timed_loop(lambda i: enc.encode(planes[0], planes[1], planes[2], W, H, row0, nrows, y0, False, stream=sp), 2, 5)
        # the seven phases, three instrumented steps (each synchronised), max over ranks of the mean
        enc.phase_events = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
        acc = None
        for _ in range(3):
            enc.encode(planes[0], planes[1], planes[2], W, H, row0, nrows, y0, False, stream=sp)
            sync_all()
            pm = enc.phase_ms()
            acc = pm if acc is None else {k: acc[k] + v for k, v in pm.items()}
        enc.phase_events = None
        phases = {k: rank_max(v / 3) for k, v in acc.items()}
        seg, bits = enc.result()
        sha_sharded = hashlib.sha256(seg).hexdigest() if rank == 0 else None
        sha_single = None
        if rank == 0:
            # the same pixels encoded by this GPU alone (the reference itself cannot: `int size = W*H*3` overflows, DESIGN.md 6)
            del planes
            torch.cuda.empty_cache()
            full = torch.empty((3, H, W), dtype=torch.uint8, device="cuda")
            ctx.synth_rows_dev(full[0], full[1], full[2], W, 0, H, frame=0, family=args.family, stream=sp)
            one = torch.zeros(cap, dtype=torch.uint8, device="cuda")
            nb1 = torch.zeros(1, dtype=torch.int64, device="cuda")
            ctx.encode_batch_dev(full[0], full[1], full[2], W, H, 1, False, one, cap, nb1, None, stream=sp)
            torch.cuda.synchronize()
            n1 = int(nb1.item())
            sha_single = hashlib.sha256(one[:n1].cpu().numpy().tobytes()).hexdigest() if n1 > 0 else "overflow"
            del full, one
        dist.barrier()
        enc.close()
        out["c5"] = {"workload": "single 32768x32768 RGB image, encode split by MCU rows", "n_gpus": world, "scaling": "strong",
                     "value": float(W) * H / (ms * 1e-3) / 1e6, "unit": "MPix/s (encode)", "ms_per_step": ms, "steps": 5,
                     "phases_ms": phases, "stream_bytes": len(seg) if seg is not None else None,
                     "sha256_sharded": sha_sharded, "sha256_single_gpu": sha_single,
                     "byte_identical_to_single_gpu": (sha_sharded == sha_single) if rank == 0 else None}
        torch.cuda.empty_cache()
    except Exception as e:
        out["c5"] = {"error": repr(e)[:300]}

    # ---- C4 --shard: one 8192x8192 --gray image, encode + decode sharded by MCU rows ----
    try:
        W = H = 8192
        row0, nrows = shard.partition_mcu_rows((H + 15) // 16, world)[rank]
        y0, ny = shard.pixel_rows(H, row0, nrows)
        planes = torch.empty((3, ny, W), dtype=torch.uint8, device="cuda")
        ctx.synth_rows_dev(planes[0], planes[1], planes[2], W, y0, ny, frame=0, family=args.family, stream=sp)
        cap = W * H // 2
        frame = J.default_frame(W, H)
        enc = shard.ShardedEncoder(ctx, grp, cap)
        dec = shard.ShardedDecoder(ctx, grp, frame, cap)
        enc.encode(planes[0], planes[1], planes[2], W, H, row0, nrows, y0, True, stream=sp)
        seg, _ = enc.result()
        nb = torch.zeros(1, dtype=torch.int64, device="cuda")
        if rank == 0:
            nb[0] = len(seg)
            dec.scan[: len(seg)] = torch.frombuffer(bytearray(seg), dtype=torch.uint8).cuda()
        dist.broadcast(nb, src=0)
        n_scan = int(nb.item())

        def step(i):
            enc.encode(planes[0], planes[1], planes[2], W, H, row0, nrows, y0, True, stream=sp)
            dec.decode(n_scan, True, stream=sp)
        ms = timed_loop(step, 2, 8)
        res = dec.result()
        same = None
        if rank == 0:
            r1, g1, b1 = ctx.decode(seg, frame, gray=True)
            same = bool((res[0] == r1).all() and (res[1] == g1).all() and (res[2] == b1).all())
        dist.barrier()
        dec.close()
        enc.close()
        out["c4_shard"] = {"workload": "--gray 8192x8192, ONE image, encode + decode sharded by MCU rows", "n_gpus": world, "scaling": "strong",
                           "value": float(W) * H / (ms * 1e-3) / 1e6, "unit": "MPix/s", "ms_per_step": ms, "steps": 8, "stream_bytes": n_scan,
                           "decode_entropy_stage": "replicated on every rank (segment broadcast from rank 0); transform stage sharded",
                           "planes_identical_to_single_gpu_decode": same}
    except Exception as e:
        out["c4_shard"] = {"error": repr(e)[:300]}
    if own_group:
        dist.destroy_process_group()
    return out


# --dump-outputs stays under 64 MB: 12 Mi float32 decoded samples + 3 Mi float32 segment bytes + the segment lengths
DUMP_DECODED_VALUES = 12 << 20
DUMP_SEGMENT_VALUES = 3 << 20


def dump_outputs(out_dir, scan, nbytes, planes):
    """One ring slot's results, its work finished: scan [B, slot] uint8, nbytes [B] int64, planes [3, B, plane_len] uint8 on the
    device -> out_dir/{segments,segment_bytes,decoded}.npy.  An array above its budget is replaced by the values at a seeded
    sample of its positions (sorted; the same positions in every run with the same arguments)."""
    import numpy as np
    import torch

    def sample(flat, budget, seed):
        if flat.numel() > budget:
            idx = np.unique(np.random.default_rng(seed).integers(0, flat.numel(), size=budget))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        return flat.cpu().numpy().astype(np.float32)

    lengths = nbytes.cpu().numpy()
    segments = torch.cat([scan[i, : int(n)] for i, n in enumerate(lengths)])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "segments.npy"), sample(segments, DUMP_SEGMENT_VALUES, 1))
    np.save(os.path.join(out_dir, "segment_bytes.npy"), lengths.astype(np.float64))
    np.save(os.path.join(out_dir, "decoded.npy"), sample(planes.reshape(-1), DUMP_DECODED_VALUES, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="frames per GPU per step (c3)")
    ap.add_argument("--family", type=int, default=0, help="0 S-photo, 1 S-noise")
    ap.add_argument("--ring", type=int, default=None, help="distinct input/output frame sets rotated between steps")
    ap.add_argument("--width", type=int, default=None, help="c5: override the image width")
    ap.add_argument("--height", type=int, default=None, help="c5: override the image height")
    ap.add_argument("--shard", action="store_true", help="c4 under torchrun: ONE image split by MCU rows over the ranks (strong scaling)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--in-flight", type=int, default=0, help="steps in flight in the device-timed loop: step i runs on context / stream i mod F "
                    "(0 = 4 for one image per step, 2 for batches, which nearly fill the machine by themselves)")
    ap.add_argument("--e2e-lanes", type=int, default=2, help="host pipelines (encode thread + decode thread each) run side by side in the e2e measurement")
    ap.add_argument("--no-configs", action="store_true", help="skip the c3 / c5 / c4_shard measurements appended to the default line")
    ap.add_argument("--host-lengths", action="store_true", help="segment lengths through a host array between encoder and decoder (round-1 step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the segments and decoded planes of the last timed step "
                    "(rank 0) to DIR/*.npy; by-image workloads only")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    sharded = args.workload == "c5" or (args.workload == "c4" and int(os.environ.get("WORLD_SIZE", "1")) > 1 and args.shard)
    if args.dump_outputs and (args.impl == "reference" or sharded):
        ap.error("--dump-outputs covers the by-image workloads of --impl b200 (c1, c2, c3, c4 without --shard)")
    claim_stdout()
    wl = dict(WORKLOADS[args.workload])
    if args.batch:
        wl["batch"] = args.batch
    if args.impl == "reference":
        args.steps = args.steps or 5
        args.warmup = args.warmup if args.warmup is not None else 1
        return run_reference(args, wl)
    if args.workload == "c5":
        return run_sharded(args, wl)
    if sharded:
        return run_sharded_gray(args, wl)
    args.steps = args.steps or 200
    args.warmup = args.warmup if args.warmup is not None else 10
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import jpezy_b200 as J
    from jpezy_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = J.Context(local_rank)
    # a real (non-default) stream: the C ABI treats a NULL stream as "the context's own stream"
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    assert sp != 0

    W, H, B, gray = wl["W"], wl["H"], wl["batch"], wl["gray"]
    npx = W * H
    frame = J.default_frame(W, H)
    plane_len = J.plane_bytes(frame)
    in_bytes = 3 * npx * B
    out_bytes = 3 * plane_len * B
    ring = args.ring or max(2, -(-300_000_000 // (in_bytes + out_bytes)))      # > 126 MB L2 with margin
    slot = max(npx, 65536)        # bytes per image for the entropy-coded segment (1 B/px; ~0.05-0.35 B/px needed)

    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- synthetic inputs, generated on the device, checked against the host twin on one frame ----
    d_in = torch.empty((ring, 3, B, H, W), dtype=torch.uint8, device="cuda")
    d_out = torch.zeros((ring, 3, B, plane_len), dtype=torch.uint8, device="cuda")
    d_scan = torch.zeros((ring, B, slot), dtype=torch.uint8, device="cuda")
    d_nbytes = torch.zeros((ring, B), dtype=torch.int64, device="cuda")
    d_status = torch.zeros((ring, B), dtype=torch.int32, device="cuda")
    for k in range(ring):
        ctx.synth_dev(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, nimg=B, first_frame=(rank * ring + k) * B, family=args.family, stream=sp)
    torch.cuda.synchronize()
    if rank == 0:
        chk = J.synth.plane(args.family, W, min(H, 64), 0, 1)
        assert (d_in[0, 1, 0, : chk.shape[0]].cpu().numpy() == chk).all(), "device synth != host synth"

    h_nbytes = [None] * ring
    h_nb = np.zeros((ring, B), dtype=np.uint64)
    # per-slot argument tuples built once: indexing a torch tensor costs microseconds, the step is ~200 of them
    enc_args = [(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, B, gray, d_scan[k], slot, d_nbytes[k], None) for k in range(ring)]
    dec_out = [(d_out[k, 0], d_out[k, 1], d_out[k, 2], plane_len, d_status[k]) for k in range(ring)]

    # Device-resident round trip: the decoder reads the segment lengths the encoder left in device memory
    # (jpezyb200_decode_batch_dev2), sized for `bound` bytes per segment -- no host round trip inside the step.  The bound
    # comes from one synchronous pass over the ring below (the largest segment + 25 %): a segment that outgrew it would
    # report JPEZYB200_ECAPACITY in d_status, which is checked after the timed loop.  --host-lengths times the round-1
    # form (lengths read back to a host array between the encoder and the decoder).
    bound = [slot]

    def step_host(k):
        ctx.encode_batch_dev(*enc_args[k], stream=sp)
        ctx.read_sizes(enc_args[k][9], B, h_nb[k], stream=sp)
        h_nbytes[k] = h_nb[k]
        ctx.decode_batch_dev(enc_args[k][7], slot, h_nb[k], B, frame, gray, *dec_out[k], stream=sp)

    # Steps are independent (every step has its own frame of the ring), and half of a single-frame step is latency bound (the chains
    # of the entropy decoder occupy a fraction of the machine): F steps in flight -- step i on context / stream i mod F, as a
    # server that transcodes a stream of frames would run them -- fill those holes.  F = 1 is one step after the other.
    n_fly = args.in_flight if args.in_flight > 0 else (4 if B == 1 else 2)
    if args.host_lengths:
        n_fly = 1
    n_fly = max(1, min(n_fly, ring))
    fly_ctx = [ctx] + [J.Context(local_rank) for _ in range(n_fly - 1)]
    fly_stream = [stream] + [torch.cuda.Stream() for _ in range(n_fly - 1)]
    fly_sp = [x.cuda_stream for x in fly_stream]

    def step_dev(k, j=0):
        fly_ctx[j].encode_batch_dev(*enc_args[k], stream=fly_sp[j])
        fly_ctx[j].decode_batch_dev2(enc_args[k][7], slot, enc_args[k][9], bound[0], B, frame, gray, *dec_out[k], stream=fly_sp[j])

    for k in range(ring):
        step_host(k)
    bound[0] = min(slot, int(max(int(x.max()) for x in h_nbytes) * 1.25) + 4096)
    step = step_host if args.host_lengths else step_dev

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, ring)):      # every ring slot is produced at least once before timing
        step(i % ring)
    barrier()

    def timed_steps(nf):
        """K steps, nf in flight: device time between an event in front of the first and one behind the last step of every stream"""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for j in range(1, nf):
            fly_stream[j].wait_event(e0)
        for i in range(args.steps):
            if nf == 1:
                step(i % ring)
            else:
                step_dev(i % ring, i % nf)
        for j in range(1, nf):
            ev = torch.cuda.Event()
            ev.record(fly_stream[j])
            stream.wait_event(ev)
        e1.record(stream)
        barrier()
        t_ms = e0.elapsed_time(e1)
        if dist is not None:
            tt = torch.tensor([t_ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_ms = float(tt.item())
        return t_ms
    if n_fly > 1:
        for i in range(max(args.warmup, 2 * n_fly)):
            step_dev(i % ring, i % n_fly)
        barrier()
    def check_round_trip(slot_k):
        """status of every decode of the ring, segment sizes, and the PSNR of one decoded frame against its input (parity itself
        is the tests' job; this catches a step that does no work, or a segment that outgrew the bound of the device-length form)"""
        assert int(d_status.abs().sum().item()) == 0, "decode reported an error status: %s" % d_status.flatten()[:8].tolist()
        assert int((d_nbytes < 0).sum().item()) == 0, "entropy-coded segment overflowed its slot"
        a = d_in[slot_k, :, 0].reshape(3, H, W)[:, : min(H, 512)].float()
        b = d_out[slot_k, :, 0, : H * W].reshape(3, H, W)[:, : min(H, 512)].float() if (W % 16 == 0) else None
        if b is None:
            return None
        if gray:
            a = (0.299 * a[0] + 0.587 * a[1] + 0.114 * a[2]).unsqueeze(0)
            b = b[:1]
        mse = float(((a - b) ** 2).mean().item())
        val = 10.0 * math.log10(255.0 ** 2 / max(mse, 1e-9))
        assert val > (24.0 if args.family == 0 else 8.0), f"round trip PSNR {val:.1f} dB: the decoded frame is not the encoded one"
        return val

    psnr = check_round_trip(0)
    d_out.zero_()          # the timed loop has to produce the pictures again

    sampler.mark = True
    l0 = sum(c.stat(capi.STAT_KERNEL_LAUNCHES) for c in fly_ctx)
    ms = timed_steps(n_fly)
    launches = sum(c.stat(capi.STAT_KERNEL_LAUNCHES) for c in fly_ctx) - l0
    psnr_after = check_round_trip((args.steps - 1) % ring)      # the last step's output, after the timed loop
    if args.dump_outputs and rank == 0:
        k_last = (args.steps - 1) % ring
        dump_outputs(args.dump_outputs, d_scan[k_last], d_nbytes[k_last], d_out[k_last])
    value = world * B * npx * args.steps / (ms * 1e-3) / 1e6
    one_in_flight = None
    if n_fly > 1:      # the same K steps one after the other on one stream, for comparison
        ms1 = timed_steps(1)
        one_in_flight = {"value": world * B * npx * args.steps / (ms1 * 1e-3) / 1e6, "unit": "MPix/s", "ms_per_step": ms1 / args.steps}

    # ---- per-stage device times + roofline of the dominant kernel (forward transform), same ring ----
    nm = capi.num_mcus(W, H)
    d_coefs = torch.empty((ring, B, nm, 6, 64), dtype=torch.int16, device="cuda")

    def timed(fn, iters):
        for i in range(3):
            fn(i % ring)
        torch.cuda.synchronize()
        a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for i in range(iters):
            fn(i % ring)
        b2.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b2) / iters

    it = max(10, min(args.steps, 100))
    t_fwd = timed(lambda k: ctx.transform_fwd_dev(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, B, gray, d_coefs[k], stream=sp), it)
    t_ent = timed(lambda k: ctx.entropy_encode_dev(d_coefs[k], W, H, B, gray, d_scan[k], slot, d_nbytes[k], None, stream=sp), it)
    t_dent = timed(lambda k: ctx.entropy_decode_dev(d_scan[k], slot, h_nbytes[k], B, frame, d_coefs[k], d_status[k], stream=sp), it)
    t_inv = timed(lambda k: ctx.transform_inv_dev(d_coefs[k], frame, B, gray, d_out[k, 0], d_out[k, 1], d_out[k, 2], plane_len, stream=sp), it)
    sampler.mark = None
    peak, peak_src = measured_peak()
    bpp = 5.0 if gray else 6.0     # SURVEY.md 8d: 3 B/px RGB in + 3 B/px int16 coefficients out (gray: chroma coefficients constant)
    dom = ("k_fwd_transform", t_fwd) if t_fwd >= t_inv else ("k_inv_transform", t_inv)
    alg_bytes = bpp * B * npx
    achieved = alg_bytes / (dom[1] * 1e-3) / 1e9
    traffic = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        traffic = prof.get(args.workload, {}).get(dom[0])
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom[0], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                "ms_per_launch": dom[1]}
    scan_bytes = float(np.mean([x.sum() for x in h_nbytes if x is not None]))
    stages = {"fwd_transform_ms": t_fwd, "entropy_encode_ms": t_ent, "entropy_decode_ms": t_dent, "inv_transform_ms": t_inv,
              "fwd_transform_GBs": bpp * B * npx / t_fwd / 1e6, "inv_transform_GBs": bpp * B * npx / t_inv / 1e6,
              "entropy_encode_Gbit_s": scan_bytes * 8 / t_ent / 1e6, "entropy_decode_Gbit_s": scan_bytes * 8 / t_dent / 1e6,
              # scan efficiency = algorithmic bytes / bytes the kernels move (model of the passes listed in DESIGN.md 4.2):
              #   encode: algorithmic 3 B/px coefficients read + S written; moved: coefficients read twice (lengths, scatter),
              #           4 B/block of offsets written and read, un-stuffed stream zeroed + written + read twice, S written
              #   decode: algorithmic S read + 3 B/px written; moved: S read twice + written once (un-stuffing), the spans read by
              #           launch 0, launch 1 and the writing pass, 3 B/px zeroed, ~1 sector per non-zero coefficient group
              #           (taken as 3 B/px), DC fix-up 2 x 32 B per block
              "entropy_encode_scan_efficiency": (3.0 * B * npx + scan_bytes) / (6.0 * B * npx + 8.0 * B * npx / 64 * 1.5 + 5.0 * scan_bytes),
              "entropy_decode_scan_efficiency": (3.0 * B * npx + scan_bytes) / (6.0 * scan_bytes + 6.0 * B * npx + 64.0 * B * npx * 1.5 / 64),
              "scan_bytes_per_step": scan_bytes, "bits_per_pixel": scan_bytes * 8 / (B * npx),
              "encode_MPix_s": B * npx / (t_fwd + t_ent) / 1e3, "decode_MPix_s": B * npx / (t_dent + t_inv) / 1e3}

    # ---- e2e: host buffers through jpezyb200_encode / jpezyb200_decode, pinned memory, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        import ctypes as C
        L = ctx.lib
        if B == 1:
            # one image per step: the per-image host entry points, as the reference's encoder / decoder objects are used
            nh = max(2, min(ring, 4))
            hin = [[torch.empty(npx, dtype=torch.uint8).pin_memory() for _ in range(3)] for _ in range(nh)]
            for k in range(nh):
                for c in range(3):
                    hin[k][c].copy_(d_in[k % ring, c, 0].reshape(-1).cpu())
            hscan = torch.empty(max(npx * 3, 10240), dtype=torch.uint8).pin_memory()
            hout = [torch.empty(plane_len, dtype=torch.uint8).pin_memory() for _ in range(3)]
            nbytes_c, nbits_c = C.c_size_t(0), C.c_uint64(0)
            api = "jpezyb200_encode + jpezyb200_decode (host pointers, pinned)"

            def e2e_step(k):
                ctx._chk(L.jpezyb200_encode(ctx.h, hin[k][0].data_ptr(), hin[k][1].data_ptr(), hin[k][2].data_ptr(), W, H, int(gray),
                                            hscan.data_ptr(), hscan.numel(), C.byref(nbytes_c), C.byref(nbits_c)))
                ctx._chk(L.jpezyb200_decode(ctx.h, hscan.data_ptr(), nbytes_c.value, C.byref(frame), int(gray), hout[0].data_ptr(),
                                            hout[1].data_ptr(), hout[2].data_ptr(), plane_len))
                return nbytes_c.value
        else:
            # a batch per step: the pipelined host batch entry points (copies of one group overlap the kernels of the previous one)
            nh = 2
            hin = [[torch.empty((B, npx), dtype=torch.uint8).pin_memory() for _ in range(3)] for _ in range(nh)]
            for k in range(nh):
                for c in range(3):
                    hin[k][c].copy_(d_in[k % ring, c].reshape(B, npx).cpu())
            hslot = max(npx // 2, 65536)
            hscan = torch.empty((B, hslot), dtype=torch.uint8).pin_memory()
            hout = [torch.empty((B, plane_len), dtype=torch.uint8).pin_memory() for _ in range(3)]
            hnb = np.zeros(B, dtype=np.uint64)
            hst = np.zeros(B, dtype=np.int32)
            api = "jpezyb200_encode_batch + jpezyb200_decode_batch (host pointers, pinned, 3-stream pipeline)"

            def e2e_step(k):
                ctx.encode_batch(hin[k][0], hin[k][1], hin[k][2], W, H, B, gray, hscan, hslot, hnb)
                ctx.decode_batch(hscan, hslot, hnb, B, frame, gray, hout[0], hout[1], hout[2], plane_len, hst)
                assert not hst.any()
                return int(hnb.sum())
        for i in range(3):
            e2e_step(i % nh)
        n_e2e = max(3, min(args.steps, 20))
        barrier()
        t0 = time.perf_counter()
        sb = 0
        for i in range(n_e2e):
            sb += e2e_step(i % nh)
        torch.cuda.synchronize()
        dt_seq = time.perf_counter() - t0
        sb /= n_e2e

        # The same calls as a two-stage pipeline: while step i is decoded (device -> host is the long copy), step i + 1 is
        # encoded (host -> device is the long copy) by a second host thread on a second context -- PCIe is full duplex and
        # a context is used by one thread at a time (SURVEY.md 8b "Threading").  Every step still carries its own
        # host-to-device copy of the input planes and device-to-host copy of the decoded planes.  --e2e-lanes L runs L such
        # pipelines side by side (steps i = lane mod L; 2 L contexts, 2 L host threads), the way a transcoding host with several
        # worker threads would: while one lane's kernels run, another lane's copies keep the two copy engines busy.
        n_lanes = max(1, args.e2e_lanes)
        n_pipe = 2 * n_e2e

        class Lane:
            def __init__(self, k):
                self.k = k
                self.ctx_e = ctx if k == 0 else J.Context(local_rank)
                self.ctx_d = J.Context(local_rank)
                self.hscan2 = [hscan if k == 0 else torch.empty_like(hscan).pin_memory(), torch.empty_like(hscan).pin_memory()]
                self.hout = hout if k == 0 else [torch.empty_like(x).pin_memory() for x in hout]
                self.nb2 = [C.c_size_t(0), C.c_size_t(0)]
                self.nbits = C.c_uint64(0)
                self.hnb2 = [np.zeros(B, dtype=np.uint64), np.zeros(B, dtype=np.uint64)]
                self.hst = np.zeros(B, dtype=np.int32)
                # two scan buffers between the stages: the encoder may run up to two steps ahead of the decoder
                self.filled = [threading.Semaphore(0), threading.Semaphore(0)]
                self.free = [threading.Semaphore(1), threading.Semaphore(1)]

            def enc_stage(self, i, j):        # step i of the run, j-th step of this lane
                src = hin[i % nh]
                if B == 1:
                    self.ctx_e._chk(L.jpezyb200_encode(self.ctx_e.h, src[0].data_ptr(), src[1].data_ptr(), src[2].data_ptr(), W, H, int(gray),
                                                       self.hscan2[j & 1].data_ptr(), self.hscan2[j & 1].numel(), C.byref(self.nb2[j & 1]),
                                                       C.byref(self.nbits)))
                else:
                    self.ctx_e.encode_batch(src[0], src[1], src[2], W, H, B, gray, self.hscan2[j & 1], hslot, self.hnb2[j & 1])

            def dec_stage(self, j):
                if B == 1:
                    self.ctx_d._chk(L.jpezyb200_decode(self.ctx_d.h, self.hscan2[j & 1].data_ptr(), self.nb2[j & 1].value, C.byref(frame),
                                                       int(gray), self.hout[0].data_ptr(), self.hout[1].data_ptr(), self.hout[2].data_ptr(),
                                                       plane_len))
                else:
                    self.ctx_d.decode_batch(self.hscan2[j & 1], hslot, self.hnb2[j & 1], B, frame, gray, self.hout[0], self.hout[1],
                                            self.hout[2], plane_len, self.hst)
                    assert not self.hst.any()

        lanes = [Lane(k) for k in range(n_lanes)]
        errs = []

        def steps_of(lane):
            return list(range(lane.k, n_pipe, n_lanes))

        def dec_worker(lane):
            try:
                torch.cuda.set_device(local_rank)
                for j, _ in enumerate(steps_of(lane)):
                    lane.filled[j & 1].acquire()
                    if errs:
                        return
                    lane.dec_stage(j)
                    lane.free[j & 1].release()
            except Exception as ex:      # noqa: BLE001
                errs.append(ex)
                for sem in lane.free:
                    sem.release()

        def enc_worker(lane):
            try:
                torch.cuda.set_device(local_rank)
                for j, i in enumerate(steps_of(lane)):
                    lane.free[j & 1].acquire()
                    if errs:
                        break
                    lane.enc_stage(i, j)
                    lane.filled[j & 1].release()
            except Exception as ex:      # noqa: BLE001
                errs.append(ex)
                for sem in lane.filled:
                    sem.release()

        for lane in lanes:               # warm every context
            lane.enc_stage(0, 0), lane.dec_stage(0)
        barrier()
        ths = [threading.Thread(target=dec_worker, args=(lane,)) for lane in lanes] + \
              [threading.Thread(target=enc_worker, args=(lane,)) for lane in lanes[1:]]
        t0 = time.perf_counter()
        for th in ths:
            th.start()
        enc_worker(lanes[0])
        for th in ths:
            th.join()
        torch.cuda.synchronize()
        dt_pipe = time.perf_counter() - t0
        if errs:
            raise errs[0]
        for lane in lanes:
            lane.ctx_d.close()
            if lane.k:
                lane.ctx_e.close()
        dts = [dt_seq, dt_pipe]
        if dist is not None:
            t = torch.tensor(dts, device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dts = [float(x) for x in t.tolist()]
        v_seq = world * B * npx * n_e2e / dts[0] / 1e6
        v_pipe = world * B * npx * n_pipe / dts[1] / 1e6
        e2e = {"value": v_pipe, "unit": "MPix/s", "h2d_bytes_per_step": int(3 * npx * B + sb),
               "d2h_bytes_per_step": int(sb + 3 * plane_len * B), "steps": n_pipe,
               "api": api + "; two-stage host pipeline: step i+1 is encoded (one context and host thread) while step i is decoded "
                            "(a second context and host thread), every step with its own H2D and D2H copies; %d such pipelines "
                            "side by side (--e2e-lanes)" % n_lanes, "lanes": n_lanes,
               "one_call_after_the_other": {"value": v_seq, "unit": "MPix/s", "steps": n_e2e}}
        # The ceiling of this figure on this host: the step's copies alone (its host-to-device bytes and its device-to-host
        # bytes, pinned, in opposite directions at the same time on two streams, no kernels), all ranks at once.  A step can
        # not be faster than its copies; e2e.frac_of_ceiling says how much of what the PCIe links / the host memory give is
        # reached (tools/pcie_probe.py is the same measurement as a stand-alone probe).
        try:
            s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
            up_src = [t_.reshape(-1) for t_ in hin[0]]
            up_dst = [torch.empty(x.numel(), dtype=torch.uint8, device="cuda") for x in up_src]
            dn_dst = [t_.reshape(-1) for t_ in hout]
            dn_src = [torch.empty(x.numel(), dtype=torch.uint8, device="cuda") for x in dn_dst]
            n_probe = 10

            def probe():
                with torch.cuda.stream(s_up):
                    for a_, b_ in zip(up_dst, up_src):
                        a_.copy_(b_, non_blocking=True)
                with torch.cuda.stream(s_dn):
                    for a_, b_ in zip(dn_dst, dn_src):
                        a_.copy_(b_, non_blocking=True)
            for _ in range(2):
                probe()
            barrier()
            t0 = time.perf_counter()
            for _ in range(n_probe):
                probe()
            torch.cuda.synchronize()
            dt_probe = time.perf_counter() - t0
            if dist is not None:
                tp = torch.tensor([dt_probe], device="cuda", dtype=torch.float64)
                dist.all_reduce(tp, op=dist.ReduceOp.MAX)
                dt_probe = float(tp.item())
            ceil_v = world * B * npx * n_probe / dt_probe / 1e6
            e2e["ceiling"] = {"value": ceil_v, "unit": "MPix/s",
                              "how": "copies of one step only: %d B host-to-device and %d B device-to-host per rank, pinned, concurrently on two "
                                     "streams, %d ranks at once" % (sum(x.numel() for x in up_src), sum(x.numel() for x in dn_dst), world),
                              "h2d_GBs_per_rank": sum(x.numel() for x in up_src) * n_probe / dt_probe / 1e9,
                              "d2h_GBs_per_rank": sum(x.numel() for x in dn_dst) * n_probe / dt_probe / 1e9}
            e2e["frac_of_ceiling"] = v_pipe / ceil_v
        except Exception as ex:
            e2e["ceiling"] = {"error": repr(ex)[:200]}

    sampler.stop_flag = True
    clocks = sampler.summary()

    # ---- CPU baseline: the oracle port on the host cores, rank 0 at N=1 only, bounded sample ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        timer, kind = cpu_arm()
        rows = min(H, 1024)
        r, g, b = (d_in[0, c, 0, :rows].cpu().numpy() for c in range(3))
        wall1, te1, td1 = timer(r, g, b, W, rows, gray, 1, 1)
        cores = os.cpu_count() or 1
        wallc, _, _ = timer(r, g, b, W, rows, gray, 1, cores)
        px = float(W) * rows
        cpu = {"value": px / wall1 / 1e6, "unit": "MPix/s", "cores": 1, "kind": kind,
               "sample": "%dx%d band (first %d rows) of one workload frame, 1 round trip, encode()+decode(), PNM I/O excluded" % (W, rows, rows),
               "encode_MPix_s": px / te1 / 1e6, "decode_MPix_s": px / td1 / 1e6,
               "all_cores": {"cores": cores, "value": px * cores / wallc / 1e6, "how": "one single-threaded instance per core"}}

    # ---- the other BASELINE.json configurations (C3 by image, C5 / C4 by MCU rows), same process, same ranks ----
    configs = None
    if args.workload == "c2" and not args.no_configs:
        del d_in, d_out, d_scan, d_coefs
        torch.cuda.empty_cache()
        configs = extra_configs(args, ctx, dist, rank, local_rank, world)

    if rank == 0:
        line = {"metric": "encode+decode MPix/s", "value": value, "unit": "MPix/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32/f64", "data": "synthetic",
                "config": {"workload": wl["name"], "width": W, "height": H, "batch_per_gpu": B, "gray": gray,
                           "family": "S-photo" if args.family == 0 else "S-noise",
                           "l2": "ring of %d distinct input/output frame sets (%.0f MB) rotated between steps; > 126 MB L2" % (
                               ring, ring * (in_bytes + out_bytes) / 1e6),
                           "sharding": "by image, no data-path collective",
                           "steps_in_flight": "%d (step i runs on context / stream i mod %d; device time from an event in front of the first "
                                              "to one behind the last step of every stream)" % (n_fly, n_fly) if n_fly > 1 else "1 (one step after the other on one stream)"},
                "steps_in_flight": n_fly, "one_step_in_flight": one_in_flight,
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "stages": stages, "configs": configs, "roundtrip_psnr_db": psnr, "roundtrip_psnr_db_after_timed_loop": psnr_after,
                "segment_lengths": "host array (read back between encoder and decoder)" if args.host_lengths else "device memory (jpezyb200_decode_batch_dev2, sized for %d bytes per segment)" % bound[0]}
        emit(line)
    if dist is not None:
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
