"""-m gpu tests of the forward transform on adversarial pixels (tests/pixel_build.py): exact quantisation ties in luma and
chroma, 32-MCU tiles at 1023, 1024, 1025 and 1152 coefficients certainly in the fix-up queue (kFixCap = 1024: the last two
take the overflow branch), blocks at 0.1 to 4 guard bands from a multiple of q and around |w| = 1 at every AC position of
both classes, every zig-zag group mask of the fused entropy coders' side information with all-black, all-white and DC-only
blocks, and ragged frames whose last column and row alternate 0/255.  Every encode route that takes pixels must give the
reference encoder's coefficients or segment:

- transform_fwd_dev, production kernel and the FP64 validation kernel (JPEZYB200_OPT_TRANSFORM = 1): oracle.coefs;
- jpezyb200_encode, encode_batch_dev and the host encode_batch (fused, reading the side information): oracle.encode;
- the same at restart intervals of 1 and 7 MCUs: oracle.scan_from_coefs of the oracle's coefficients;
- encode_optimized / encode_batch_optimized_dev: tables from the symbol counts of the oracle's coefficients, and the
  segment that jpeg_build.encode_scan writes with the device's tables;
- shard.encode_sharded_local with 2 to 4 emulated ranks: oracle.encode.

Device outputs land in Guarded buffers."""
import numpy as np
import pytest
import torch

import jpezy_b200 as J
from jpezy_b200 import capi, shard
from jpezy_b200.capi import OPT_RESTART_INTERVAL, OPT_TRANSFORM, STAT_GUARD_FWD, num_mcus
from gpu_util import Guarded, to_dev
from jpeg_build import Huff, encode_scan
from test_huffopt_gpu import check_tables
from test_pixel_build import sweep_gaps
import pixel_build as P

pytestmark = pytest.mark.gpu

HB = capi.HUFF_TABLES_BYTES
RAGGED = ([(16 + r, 16 + (r * 7) % 16) for r in range(16)] + [(W, 24) for W in (1, 15, 17, 511, 513, 527, 528)] +
          [(W, H) for W, H in ((600, 1), (600, 9), (528, 16), (33, 16))])


@pytest.fixture(scope="module")
def ties():
    return P.ties_image(21)


@pytest.fixture(scope="module")
def masks():
    return P.mask_image(22)


@pytest.fixture(scope="module")
def queue():
    return P.queue_image(23)


@pytest.fixture(scope="module")
def sweep():
    return P.sweep_image(24)


def stream():
    return torch.cuda.current_stream().cuda_stream


def dev_coefs(ctx, imgs, W, H, gray, fp64=False):
    """transform_fwd_dev of a batch into a guarded buffer -> [nimg, nmcu, 6, 64]"""
    n = len(imgs)
    d = to_dev(np.stack([np.stack(p) for p in imgs], 1))      # [3][n][H][W]
    out = Guarded(n * num_mcus(W, H) * 384, torch.int16, fill=-12345, offset=32)
    torch.cuda.synchronize()
    try:
        ctx.set_option(OPT_TRANSFORM, int(fp64))
        ctx.transform_fwd_dev(d[0], d[1], d[2], W, H, n, gray, out.view, stream=stream())
        torch.cuda.synchronize()
    finally:
        ctx.set_option(OPT_TRANSFORM, 0)
    assert out.intact()
    return out.view.cpu().numpy().reshape(n, -1, 6, 64)


def batch_dev(ctx, imgs, W, H, gray, optimized=False):
    """encode_batch_dev / encode_batch_optimized_dev into guarded buffers -> ([segment], [HuffTables] or None)"""
    n = len(imgs)
    d = to_dev(np.stack([np.stack(p) for p in imgs], 1))
    slot = max(W * H * 3, 10240)
    scan = Guarded(n * slot, torch.uint8, offset=16)
    nbytes = Guarded(n, torch.int64)
    ht = Guarded(n * HB, torch.uint8) if optimized else None
    torch.cuda.synchronize()
    if optimized:
        ctx.encode_batch_optimized_dev(d[0], d[1], d[2], W, H, n, gray, scan.view, slot, ht.view, nbytes.view, stream=stream())
    else:
        ctx.encode_batch_dev(d[0], d[1], d[2], W, H, n, gray, scan.view, slot, nbytes.view, stream=stream())
    torch.cuda.synchronize()
    assert scan.intact() and nbytes.intact() and (ht is None or ht.intact())
    s, nb = scan.view.cpu().numpy(), nbytes.view.cpu().numpy()
    segs = [s[i * slot: i * slot + nb[i]].tobytes() for i in range(n)]
    return segs, ([J.huff_tables(ht.view[i * HB:(i + 1) * HB]) for i in range(n)] if optimized else None)


def host_batch(ctx, imgs, W, H, gray):
    n = len(imgs)
    r, g, b = (np.ascontiguousarray(np.stack([p[c] for p in imgs])) for c in range(3))
    slot = max(W * H * 3, 10240)
    scans = np.zeros((n, slot), np.uint8)
    nbytes = np.zeros(n, np.uint64)
    ctx.encode_batch(r, g, b, W, H, n, gray, scans, slot, nbytes)
    return [scans[i, :int(nbytes[i])].tobytes() for i in range(n)]


def opt_segment(coefs, ht):
    """the segment jpeg_build writes for the oracle's coefficients with the device's four tables"""
    h = lambda t: Huff(list(t.bits), list(t.vals[:sum(t.bits)]))
    return encode_scan(np.asarray(coefs).reshape(-1, 64), "420", {c: (h(ht[0][c]), h(ht[1][c])) for c in (0, 1)})


def check_routes(ctx, oracle, imgs, W, H, gray, ranks=(2, 3)):
    """every pixel route against the reference on a batch of images -> the oracle's coefficients"""
    want = np.stack([oracle.coefs(*p, W, H, gray=gray) for p in imgs])
    for fp64 in (False, True):
        got = dev_coefs(ctx, imgs, W, H, gray, fp64)
        bad = np.argwhere(got != want)
        assert bad.size == 0, "fp64=%d: %d mismatches, first (img, mcu, blk, zz) %s" % (fp64, len(bad), bad[:4].tolist())
    scans = [oracle.encode(*p, W, H, gray=gray, scan_only=True) for p in imgs]
    for i, p in enumerate(imgs):
        assert ctx.encode(*p, W, H, gray=gray)[0] == scans[i]
    assert batch_dev(ctx, imgs, W, H, gray)[0] == scans
    assert host_batch(ctx, imgs, W, H, gray) == scans
    for R in (1, 7):
        rscans = [oracle.scan_from_coefs(c, restart_interval=R) for c in want]
        try:
            ctx.set_option(OPT_RESTART_INTERVAL, R)
            assert ctx.encode(*imgs[0], W, H, gray=gray)[0] == rscans[0]
            assert batch_dev(ctx, imgs, W, H, gray)[0] == rscans
        finally:
            ctx.set_option(OPT_RESTART_INTERVAL, 0)
    segs, hts = batch_dev(ctx, imgs, W, H, gray, optimized=True)
    for i, p in enumerate(imgs):
        seg, nbits, ht = ctx.encode_optimized(*p, W, H, gray=gray)
        assert nbits == check_tables(ht, want[i])
        assert seg == opt_segment(want[i], ht) == segs[i] and bytes(hts[i]) == bytes(ht)
    VU = (H + 15) // 16
    for n in ranks:
        if VU < n:
            continue
        ctxs = [ctx] + [J.Context(0) for _ in range(n - 1)]
        try:
            planes = tuple(to_dev(x.reshape(H, W)) for x in imgs[0])
            got, _ = shard.encode_sharded_local(ctxs, planes, W, H, gray=gray)
            assert got == scans[0], "%d ranks" % n
        finally:
            for c in ctxs[1:]:
                c.close()
    return want


# ---- exact ties ------------------------------------------------------------------------------------------------------------
def test_ties_every_route(ctx, oracle, ties):
    r, g, b, W, H = ties
    check_routes(ctx, oracle, [(r, g, b)], W, H, False)


def test_ties_gray(ctx, oracle, ties):
    r, g, b, W, H = ties
    check_routes(ctx, oracle, [(r, g, b)], W, H, True, ranks=(2,))


def test_ties_reach_the_exact_tier_on_both_kernels(ctx, oracle, ties):
    r, g, b, W, H = ties
    _, raw = oracle.coefs(r, g, b, W, H, want_raw=True)
    d = P.certify(raw)
    n_ac = int((d < 1e-6).sum())
    cls = (np.arange(6) >= 4).astype(np.int64)
    w = raw / P.Q[cls][None]
    k = np.round(w)
    n_all = int(((k != 0) & (np.abs(raw - k * P.Q[cls][None]) < 1e-7)).sum())      # the FP64 kernel also checks the DC
    assert n_ac >= 5 * 4 * 8 + 5 * 2 * 8                                            # five in every tie block
    # the production kernel counts its tier-3 evaluations, the FP64 kernel every coefficient within 1e-6 of a multiple
    for fp64, want in ((False, n_ac), (True, n_all)):
        before = ctx.stat(STAT_GUARD_FWD)
        dev_coefs(ctx, [(r, g, b)], W, H, False, fp64)
        assert ctx.stat(STAT_GUARD_FWD) - before == want, "fp64=%d" % fp64


# ---- the fix-up queue at and past its capacity ------------------------------------------------------------------------------
def exact_counts(raw, ac_only):
    """coefficients within 1e-7 of a non-zero multiple of q, per 32-MCU tile (one MCU row of the queue image)"""
    cls = (np.arange(6) >= 4).astype(np.int64)
    q = P.Q[cls][None]
    k = np.round(raw / q)
    ex = (k != 0) & (np.abs(raw - k * q) < 1e-7)
    if ac_only:
        ex[:, :, 0] = False
    return ex.reshape(len(P.QUEUE_COUNTS), -1).sum(1)


def test_queue_tiles_certified_and_counted(ctx, oracle, queue):
    r, g, b, W, H = queue
    _, raw = oracle.coefs(r, g, b, W, H, want_raw=True)
    sure, unsure = P.queued(P.certify(raw))
    assert not unsure.any()
    assert sure.reshape(len(P.QUEUE_COUNTS), -1).sum(1).tolist() == list(P.QUEUE_COUNTS)
    ac, every = exact_counts(raw, True), exact_counts(raw, False)
    assert ac.tolist() == list(P.QUEUE_COUNTS)
    # production kernel: one tier-3 evaluation per queued tie; a tile past 1024 entries re-evaluates every coefficient
    # exactly, so its DC ties count too.  FP64 kernel: every coefficient within 1e-6 of a multiple.
    want_prod = int(sum(e if c > 1024 else a for a, e, c in zip(ac, every, P.QUEUE_COUNTS)))
    for fp64, want in ((False, want_prod), (True, int(every.sum()))):
        before = ctx.stat(STAT_GUARD_FWD)
        got = dev_coefs(ctx, [(r, g, b)], W, H, False, fp64)
        assert ctx.stat(STAT_GUARD_FWD) - before == want, "fp64=%d" % fp64
        assert (got[0] == oracle.coefs(r, g, b, W, H)).all()


def test_queue_tiles_every_route(ctx, oracle, queue):
    r, g, b, W, H = queue
    check_routes(ctx, oracle, [(r, g, b)], W, H, False, ranks=(2, 3, 4))


# ---- guard-band sweep ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gray", [False, True])
def test_sweep_every_route(ctx, oracle, sweep, gray):
    r, g, b, W, H = sweep
    if not gray:
        _, raw = oracle.coefs(r, g, b, W, H, want_raw=True)
        assert not sweep_gaps(raw)
    check_routes(ctx, oracle, [(r, g, b)], W, H, gray, ranks=(2, 4))


# ---- side-information masks ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("gray", [False, True])
def test_every_group_mask(ctx, oracle, masks, gray):
    r, g, b, W, H = masks
    want = check_routes(ctx, oracle, [(r, g, b)], W, H, gray, ranks=(2, 3, 4))[0]
    c = want.reshape(-1, 6, 64).copy()
    c[:, :, 0] = 0
    seen = set(((c.reshape(-1, 6, 8, 8) != 0).any(3).astype(np.int64) @ (1 << np.arange(8))).reshape(-1).tolist())
    assert seen == set(range(256))
    assert want[..., 0].min() <= -63 and want[..., 0].max() >= 63


# ---- ragged edges ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,H", RAGGED)
def test_ragged_edges(ctx, oracle, W, H):
    imgs = [P.ragged_image(1000 * W + H + k, W, H) for k in range(3)]
    check_routes(ctx, oracle, imgs, W, H, False, ranks=())


@pytest.mark.parametrize("W,H", [(527, 40), (513, 33)])
def test_ragged_edges_gray_and_sharded(ctx, oracle, W, H):
    imgs = [P.ragged_image(7 * W + H + k, W, H) for k in range(3)]
    check_routes(ctx, oracle, imgs, W, H, True, ranks=(2, 3))
    check_routes(ctx, oracle, imgs[:1], W, H, False, ranks=(2, 3))
