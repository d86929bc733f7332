"""What restart intervals (JPEZYB200_OPT_RESTART_INTERVAL) cost and buy on the device-resident path: encode
(jpezyb200_encode_batch_dev) and decode (jpezyb200_decode_batch_dev2, lengths kept on the device) timed with CUDA events on the
launching stream, per interval, on C2 (one 3840x2160 frame) and C3 (64 1920x1080 frames) in S-photo and S-noise.

Inputs rotate through a ring larger than L2; the intervals alternate within every round, so drift of the clocks or of other
work on the machine spreads over all of them.  Every decode is checked against the restart-less decode of the same frames.

usage: python tools/restart_bench.py [--rounds 20] [--workloads c2,c3] [--families 0,1] [--intervals 0,1,4,16,row]
prints the card, its power limit and one JSON line per (workload, family, interval): median and min microseconds of the encode
and of the decode, segment bytes per step and their ratio to interval 0"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {"c2": (3840, 2160, 1), "c3": (1920, 1080, 64)}
L2_BYTES = 126 << 20


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi not available"
    return name, q


def run(ctx, W, H, nimg, family, intervals, rounds):
    import numpy as np
    import torch
    import jpezy_b200 as J
    from jpezy_b200 import capi

    npx = W * H
    ring = max(2, -(-2 * L2_BYTES // (3 * npx * nimg)))     # input sets: together more than twice the L2
    # a stream of its own: stream 0 would mean the context's own stream to the library, and the events would time nothing
    st = torch.cuda.Stream()
    sp = st.cuda_stream
    rgb = torch.empty((ring, 3, nimg * npx), dtype=torch.uint8, device="cuda")
    for k in range(ring):
        ctx.synth_dev(rgb[k, 0], rgb[k, 1], rgb[k, 2], W, H, nimg, first_frame=k * nimg, family=family, stream=sp)
    slot = (3 * npx // 16 + 1) * 16
    scan = torch.zeros((ring, nimg, slot), dtype=torch.uint8, device="cuda")
    nbytes = torch.zeros((ring, nimg), dtype=torch.int64, device="cuda")
    frame = J.default_frame(W, H)
    need = capi.plane_bytes(frame)
    out = torch.empty((3, nimg * need), dtype=torch.uint8, device="cuda")
    ref = {}
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize()   # (the buffers were zeroed on torch's stream)
    t_enc = {R: [] for R in intervals}
    t_dec = {R: [] for R in intervals}
    seg = {R: 0 for R in intervals}

    def step(k, R, timed):
        ctx.set_option(capi.OPT_RESTART_INTERVAL, R)
        frame.restart_interval = R
        e[0].record(st)
        ctx.encode_batch_dev(rgb[k, 0], rgb[k, 1], rgb[k, 2], W, H, nimg, False, scan[k], slot, nbytes[k], None, stream=sp)
        e[1].record(st)
        ctx.decode_batch_dev2(scan[k], slot, nbytes[k], slot, nimg, frame, False, out[0], out[1], out[2], need, None, stream=sp)
        e[2].record(st)
        torch.cuda.synchronize()
        if timed:
            t_enc[R].append(e[0].elapsed_time(e[1]) * 1e3)
            t_dec[R].append(e[1].elapsed_time(e[2]) * 1e3)
        if (nbytes[k] < 0).any():
            raise RuntimeError("a segment did not fit its slot")
        if k not in ref:
            ref[k] = out.clone() if R == 0 else None
        if ref[k] is not None and not torch.equal(out, ref[k]):
            raise RuntimeError("interval %d decodes to other planes than interval 0" % R)
        return int(nbytes[k].sum())

    for k in range(ring):                       # warm-up: every shape, every interval; interval 0 first (the reference planes)
        for R in intervals:
            step(k, R, False)
    for rnd in range(rounds):
        k = rnd % ring
        order = intervals[rnd % len(intervals):] + intervals[: rnd % len(intervals)]
        for R in order:
            b = step(k, R, True)
            if rnd < ring:
                seg[R] += b
    ctx.set_option(capi.OPT_RESTART_INTERVAL, 0)
    nsets = min(rounds, ring)
    res = []
    for R in intervals:
        res.append(dict(interval=R, enc_us_median=float(np.median(t_enc[R])), enc_us_min=float(np.min(t_enc[R])),
                        dec_us_median=float(np.median(t_dec[R])), dec_us_min=float(np.min(t_dec[R])),
                        bytes_per_step=seg[R] / nsets, bytes_vs_0=seg[R] / seg[intervals[0]] if seg[intervals[0]] else None))
    del rgb, scan, out, ref
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--workloads", default="c2,c3")
    ap.add_argument("--families", default="0,1")
    ap.add_argument("--intervals", default="0,1,4,16,row", help="MCUs per interval; 'row' = one MCU row; 0 must come first")
    a = ap.parse_args()
    if a.rounds < 1:
        ap.error("--rounds must be at least 1")
    import torch
    import jpezy_b200 as J

    if not torch.cuda.is_available():
        sys.exit("restart_bench.py needs a CUDA device")
    torch.cuda.init()
    name, smi = card()
    print("card: %s | nvidia-smi (name, power limit, max SM clock): %s" % (name, smi), flush=True)
    ctx = J.Context(0)
    for wl in a.workloads.split(","):
        W, H, nimg = WORKLOADS[wl]
        ivs = [(W + 15) // 16 if s == "row" else int(s) for s in a.intervals.split(",")]
        if ivs[0] != 0:
            ap.error("the first interval must be 0 (the reference)")
        for fam in (int(f) for f in a.families.split(",")):
            for r in run(ctx, W, H, nimg, fam, ivs, a.rounds):
                print(json.dumps(dict(workload=wl, family=fam, W=W, H=H, nimg=nimg, **r)), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
