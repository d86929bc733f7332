"""-m gpu: the low-frequency class of k_inv_transform2 -- warps whose blocks have nothing beyond zig-zag position 2, evaluated as a
separable sum with their own guard band (tools/lowfreq_idct_error_bound.py) -- against the reference decoder's pixel stage, on
the per-stage path (transform_inv_dev, DC inside the blocks) and on the fused decode (dense DC array).  Bar: zero differing
samples.  Warps are 4 block pairs: luma of two MCUs, or chroma of four, of an 8-MCU tile."""
import math

import numpy as np
import pytest
import torch

from jpezy_b200 import capi
from gpu_util import Guarded
from test_inverse_reference_gpu import EAGAIN, check_planes, frame_for, geometry, qtables, reference, run_inverse, scans, upload_scans

pytestmark = pytest.mark.gpu

KINDS = ["random", "ties", "negative", "dc_mix", "wide", "mixed3", "mixed7", "mixed8"]


def lowfreq(kind, nmcu, q, seed):
    """[nmcu, 6, 64] 4:2:0 zig-zag coefficients with nothing beyond zig-zag position 2 (|F| <= 1023), except for "mixedP": one
    block in about sixteen also has a coefficient at zig-zag position P, which moves its warp off the class"""
    rng = np.random.default_rng(seed)
    c = np.zeros((nmcu, 6, 64), np.int32)
    flat = c.reshape(-1, 64)
    n = flat.shape[0]
    comp = np.tile([0, 0, 0, 0, 1, 2], nmcu)
    if kind in ("random", "mixed3", "mixed7", "mixed8"):
        flat[:, 0] = rng.integers(-1023, 1024, n)
        flat[:, 1:3] = rng.integers(-200, 201, (n, 2))
        if kind != "random":
            hit = rng.choice(n, max(1, n // 16), replace=False)
            flat[hit, int(kind[5:])] = rng.integers(1, 60, hit.size) * rng.choice([-1, 1], hit.size)
    elif kind == "ties":
        # F01 q01 = +-F10 q10 and DC q00 a multiple of 8: on one diagonal of the block the two cosine terms cancel and the exact
        # sample is the integer DC q00 / 8 + 128, which only the reference's FP64 rounding decides
        for i in range(n):
            qq = q[comp[i]]
            g = math.gcd(int(qq[1]), int(qq[8]))
            k = int(rng.integers(1, 1023 // (max(qq[1], qq[8]) // g) + 1))
            flat[i, 0] = 8 * int(rng.integers(-127, 128))
            flat[i, 1] = k * int(qq[8]) // g * int(rng.choice([-1, 1]))
            flat[i, 2] = k * int(qq[1]) // g
    elif kind == "negative":                 # most samples below zero, where the reference's truncation is not floor
        flat[:, 0] = rng.integers(-1023, -300, n)
        flat[:, 1:3] = rng.integers(-100, 101, (n, 2))
    elif kind == "dc_mix":                   # DC-only blocks inside class warps (two in three)
        flat[:, 0] = rng.integers(-1023, 1024, n)
        flat[:, 1:3] = rng.integers(-50, 51, (n, 2)) * (rng.random((n, 1)) < 1 / 3)
    elif kind == "wide":                     # |AC| up to 1023: with 16-bit tables the samples leave the int16 range
        flat[:, 0] = rng.integers(-1023, 1024, n)
        flat[:, 1:3] = rng.integers(-1023, 1024, (n, 2))
    assert np.abs(c).max() <= 1023
    return c


def tables_for(oracle, kind):
    if kind == "wide":
        return qtables(oracle, "bits16")
    return qtables(oracle, {"random": "annexk", "ties": "distinct", "negative": "ones", "dc_mix": "all255"}.get(kind, "annexk"))


# 13 x 8 MCUs: a ragged last tile (5 of 8 MCUs) and H % 16 != 0; 16 x 3 MCUs: whole tiles
GEOMS = [(200, 120), (256, 48)]


@pytest.mark.parametrize("gray", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_lowfreq_per_stage_matches_reference(ctx, oracle, kind, gray):
    q = tables_for(oracle, kind)
    for gi, (W, H) in enumerate(GEOMS):
        _, _, nmcu, _ = geometry(W, H, "420")
        cs = [lowfreq(kind, nmcu, q, seed=100 * KINDS.index(kind) + 10 * gi + i) for i in range(3)]
        frame = frame_for(W, H, "420", q)
        before = ctx.stat(capi.STAT_GUARD_INV)
        got = run_inverse(ctx, cs, frame, gray, "inv2")
        for i in range(3):
            check_planes(got[i], reference(oracle, cs[i], W, H, "420", q, gray), "%s %dx%d gray %d image %d" % (kind, W, H, gray, i))
        if kind in ("ties", "wide"):          # guard-band hits decided in the reference's order / tiles on the exact-order route
            assert ctx.stat(capi.STAT_GUARD_INV) > before


def test_lowfreq_ties_hit_the_guard_band(ctx, oracle):
    """without DC-only blocks or wide samples, the statistic moves only through samples inside the guard band"""
    q = qtables(oracle, "annexk")
    W, H = 128, 16
    _, _, nmcu, _ = geometry(W, H, "420")
    c = lowfreq("ties", nmcu, q, seed=77)
    assert (c[:, :, 1:3] != 0).all()
    before = ctx.stat(capi.STAT_GUARD_INV)
    got = run_inverse(ctx, [c], frame_for(W, H, "420", q), False, "inv2")
    check_planes(got[0], reference(oracle, c, W, H, "420", q, False), "ties 128x16")
    assert ctx.stat(capi.STAT_GUARD_INV) - before >= 8 * c.shape[0] * 6 // 2


@pytest.mark.parametrize("gray", [False, True])
@pytest.mark.parametrize("kind", ["random", "ties", "negative", "dc_mix", "wide", "mixed3", "mixed8"])
def test_lowfreq_fused_decode_matches_reference(ctx, oracle, kind, gray):
    """files made from the coefficients: jpezyb200_decode and decode_batch_dev2 take the DC from the dense array"""
    q = tables_for(oracle, kind)
    W, H = GEOMS[KINDS.index(kind) % 2]
    _, _, nmcu, _ = geometry(W, H, "420")
    cs = [lowfreq(kind, nmcu, q, seed=900 + 10 * KINDS.index(kind) + i) for i in range(3)]
    frame = frame_for(W, H, "420", q)
    want = [reference(oracle, c, W, H, "420", q, gray) for c in cs]
    ss = scans(oracle, cs)
    for i in range(3):
        check_planes(ctx.decode(ss[i], frame, gray=gray), want[i], "jpezyb200_decode %s image %d" % (kind, i))
    d_scan, slot, nbytes = upload_scans(ss)
    pl = capi.plane_bytes(frame)
    out = [Guarded(3 * pl, torch.uint8, fill=0x3C) for _ in range(3)]
    st = torch.full((3,), -1, dtype=torch.int32, device="cuda")
    d_nb = torch.from_numpy(nbytes.astype(np.int64)).cuda()
    torch.cuda.synchronize()
    ctx.decode_batch_dev2(d_scan, slot, d_nb, int(nbytes.max()), 3, frame, gray, out[0].view, out[1].view, out[2].view, pl, st,
                          stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for i, s in enumerate(st.cpu().tolist()):
        assert s in (0, EAGAIN)
        if s == 0:
            check_planes([o.view[i * pl: (i + 1) * pl] for o in out], want[i], "decode_batch_dev2 %s image %d" % (kind, i))
    assert all(o.intact() for o in out)
