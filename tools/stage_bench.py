"""Times ONE stage of the device-resident path alone (CUDA events on the launching stream, inputs rotated through a ring
larger than L2): the quick loop used while tuning a kernel, and the short command ncu is pointed at.

usage: python tools/stage_bench.py [--stage fwd|inv|enc|enc_opt|dec] [--w 3840 --h 2160 --batch 1] [--family 0] [--gray] [--iters 50]
prints one JSON line: microseconds per launch, algorithmic GB/s at 6 (5 gray) B/px and the fraction of MEASURED_PEAKS.json;
enc_opt (the entropy stage with per-image optimised Huffman tables) adds the stuffed bytes of the batch with the Annex K
tables and with the optimised ones"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stage", default="fwd", choices=["fwd", "inv", "enc", "enc_opt", "dec"])
    ap.add_argument("--w", type=int, default=3840)
    ap.add_argument("--h", type=int, default=2160)
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--family", type=int, default=0)
    ap.add_argument("--gray", action="store_true")
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--variant", type=int, default=0, choices=[0, 1], help="JPEZYB200_OPT_TRANSFORM: 0 production, 1 FP64 validation kernels")
    ap.add_argument("--guesses", type=int, default=0, help="JPEZYB200_OPT_SYNC_GUESSES")
    ap.add_argument("--lib", default="", help="A/B runs: another build of libjpezy_b200.so to load instead of the in-tree one")
    a = ap.parse_args()
    import numpy as np
    import torch
    import jpezy_b200 as J
    from jpezy_b200 import capi

    if a.lib:
        capi.library_path = lambda: os.path.abspath(a.lib)
    ctx = J.Context(0)
    if a.variant:
        ctx.set_option(capi.OPT_TRANSFORM, a.variant)
    if a.guesses:
        ctx.set_option(capi.OPT_SYNC_GUESSES, a.guesses)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    W, H, B, gray = a.w, a.h, a.batch, int(a.gray)
    npx = W * H
    frame = J.default_frame(W, H)
    plane_len = J.plane_bytes(frame)
    ring = max(2, -(-300_000_000 // (6 * npx * B)))
    slot = max(npx, 65536)
    nm = capi.num_mcus(W, H)
    d_in = torch.empty((ring, 3, B, H, W), dtype=torch.uint8, device="cuda")
    d_out = torch.zeros((ring, 3, B, plane_len), dtype=torch.uint8, device="cuda")
    d_coefs = torch.empty((ring, B, nm, 6, 64), dtype=torch.int16, device="cuda")
    d_scan = torch.zeros((ring, B, slot), dtype=torch.uint8, device="cuda")
    d_nbytes = torch.zeros((ring, B), dtype=torch.int64, device="cuda")
    d_status = torch.zeros((ring, B), dtype=torch.int32, device="cuda")
    d_ht = torch.zeros((ring, B * capi.HUFF_TABLES_BYTES), dtype=torch.uint8, device="cuda")
    h_nb = np.zeros((ring, B), dtype=np.uint64)
    for k in range(ring):
        ctx.synth_dev(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, nimg=B, first_frame=k * B, family=a.family, stream=sp)
        ctx.transform_fwd_dev(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, B, gray, d_coefs[k], stream=sp)
        ctx.entropy_encode_dev(d_coefs[k], W, H, B, gray, d_scan[k], slot, d_nbytes[k], None, stream=sp)
        ctx.read_sizes(d_nbytes[k], B, h_nb[k], stream=sp)
    fns = {
        "fwd": lambda k: ctx.transform_fwd_dev(d_in[k, 0], d_in[k, 1], d_in[k, 2], W, H, B, gray, d_coefs[k], stream=sp),
        "inv": lambda k: ctx.transform_inv_dev(d_coefs[k], frame, B, gray, d_out[k, 0], d_out[k, 1], d_out[k, 2], plane_len, stream=sp),
        "enc": lambda k: ctx.entropy_encode_dev(d_coefs[k], W, H, B, gray, d_scan[k], slot, d_nbytes[k], None, stream=sp),
        "enc_opt": lambda k: ctx.entropy_encode_optimized_dev(d_coefs[k], W, H, B, gray, d_scan[k], slot, d_ht[k], d_nbytes[k], None, stream=sp),
        "dec": lambda k: ctx.entropy_decode_dev(d_scan[k], slot, h_nb[k], B, frame, d_coefs[k], d_status[k], stream=sp),
    }
    fn = fns[a.stage]
    for i in range(5):
        fn(i % ring)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(a.iters):
        fn(i % ring)
    e1.record(stream)
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / a.iters * 1e3
    extra = {}
    if a.stage == "enc_opt":   # stuffed bytes of ring slot 0, Annex K tables against optimised tables
        nb = np.zeros(B, dtype=np.uint64)
        ctx.entropy_encode_dev(d_coefs[0], W, H, B, gray, d_scan[0], slot, d_nbytes[0], None, stream=sp)
        ctx.read_sizes(d_nbytes[0], B, nb, stream=sp)
        extra["bytes_annex_k"] = int(nb.sum())
        fn(0)
        ctx.read_sizes(d_nbytes[0], B, nb, stream=sp)
        extra["bytes_optimized"] = int(nb.sum())
        extra["saving_pct"] = round(100.0 * (1 - extra["bytes_optimized"] / extra["bytes_annex_k"]), 2)
    bpp = 5.0 if gray else 6.0
    gbs = bpp * B * npx / us / 1e3
    peak = 6541.1
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    print(json.dumps({"stage": a.stage, "W": W, "H": H, "batch": B, "family": a.family, "gray": gray, "variant": a.variant, "lib": os.path.basename(a.lib),
                      "us_per_launch": round(us, 2), "GBs": round(gbs, 1),
                      "frac_of_measured_peak": round(gbs / peak, 4), "guard_fwd": ctx.stat(capi.STAT_GUARD_FWD),
                      "sync_iters": [ctx.stat(capi.STAT_SYNC_ITERS0), ctx.stat(capi.STAT_SYNC_ITERS1)], "sync_rounds": ctx.stat(capi.STAT_SYNC_ROUNDS), **extra}))


if __name__ == "__main__":
    main()
