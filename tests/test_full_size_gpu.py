"""-m gpu: parity at the sizes BASELINE.json names.

C2 (3840x2160), one C3 frame (1920x1080) and C4 (8192x8192 --gray) are small enough for the oracle: full byte / sample
parity.  For the giant-image shape (C5, 32768 wide) the oracle would take minutes, so size-independent properties are
checked on a 32768 x 1024 band and on the full-width batch: the sharded encoder equals the single-GPU encoder, entropy decode
inverts entropy encode exactly, the batch entry points equal the per-image ones, and Pillow (libjpeg) decodes our file to
within a fixed PSNR of the source image."""
import hashlib
import io

import numpy as np
import pytest
import torch

import jpezy_b200 as J
from jpezy_b200 import capi, shard

pytestmark = pytest.mark.gpu


def synth_dev(ctx, W, H, family=0, frame=0):
    d = torch.empty((3, H, W), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.synth_dev(d[0], d[1], d[2], W, H, 1, frame, family)
    torch.cuda.synchronize()
    return d


@pytest.mark.parametrize("name,W,H,gray,family", [("C2", 3840, 2160, False, 0), ("C3 frame", 1920, 1080, False, 0), ("C4", 8192, 8192, True, 0),
                                                  ("C2 S-noise", 3840, 2160, False, 1), ("C3 frame S-noise", 1920, 1080, False, 1)])
def test_full_size_byte_and_sample_parity(ctx, oracle, name, W, H, gray, family):
    # S-noise (2.5 bit/px) is the entropy stress case and the one that fills the guard-band queues of both transforms
    d = synth_dev(ctx, W, H, family=family)
    r, g, b = (d[c].cpu().numpy() for c in range(3))
    scan, nbits = ctx.encode(r, g, b, W, H, gray=gray)
    want = oracle.encode(r, g, b, W, H, gray=gray)
    assert hashlib.sha256(oracle.header(W, H, gray=gray) + scan + b"\xff\xd9").hexdigest() == hashlib.sha256(want).hexdigest()
    R, G, B = ctx.decode(scan, J.default_frame(W, H), gray=gray)
    _, _, R0, G0, B0 = oracle.decode(want, gray=gray)
    nd = int((R != R0).sum()) + int((G != G0).sum()) + int((B != B0).sum())
    assert nd == 0, "%s: %d decoded samples differ from the reference decoder" % (name, nd)


@pytest.mark.parametrize("family", [0, 1])
def test_full_size_one_chain_per_guess(ctx, oracle, family):
    # the latency form of the first synchronisation launch (JPEZYB200_OPT_SYNC_GUESSES = 1) on a whole 4K frame
    W, H = 3840, 2160
    d = synth_dev(ctx, W, H, family=family)
    r, g, b = (d[c].cpu().numpy() for c in range(3))
    want = oracle.encode(r, g, b, W, H)
    ctx.set_option(capi.OPT_SYNC_GUESSES, 1)
    try:
        R, G, B = ctx.decode(want[644:-2], J.default_frame(W, H))
    finally:
        ctx.set_option(capi.OPT_SYNC_GUESSES, 0)
    _, _, R0, G0, B0 = oracle.decode(want)
    assert int((R != R0).sum()) + int((G != G0).sum()) + int((B != B0).sum()) == 0


def test_c5_shape_properties(ctx):
    W, H = 32768, 1024                                   # a band of the 32768 x 32768 image: 2048 x 64 MCUs
    d = synth_dev(ctx, W, H)
    slot = W * H
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    out = torch.zeros(slot, dtype=torch.uint8, device="cuda")
    nb = torch.zeros(2, dtype=torch.int64, device="cuda")
    nm = capi.num_mcus(W, H)
    coefs = torch.empty((nm, 6, 64), dtype=torch.int16, device="cuda")
    with torch.cuda.stream(st):
        ctx.transform_fwd_dev(d[0], d[1], d[2], W, H, 1, False, coefs, stream=st.cuda_stream)
        ctx.entropy_encode_dev(coefs, W, H, 1, False, out, slot, nb[:1], nb[1:], stream=st.cuda_stream)
    torch.cuda.synchronize()
    n = int(nb[0].item())
    single = out[:n].cpu().numpy().tobytes()
    # (1) the sharded encoder (4 emulated ranks) writes the same stream
    ctxs = [J.Context(0) for _ in range(4)]
    try:
        got, bits = shard.encode_sharded_local(ctxs, (d[0], d[1], d[2]), W, H, dst_cap=slot)
    finally:
        for c in ctxs:
            c.close()
    assert got == single and sum(bits) == int(nb[1].item())
    # (2) entropy decode inverts entropy encode exactly, and the byte count obeys the stuffing rule
    back = torch.full((nm, 6, 64), 777, dtype=torch.int16, device="cuda")
    status = torch.full((1,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.entropy_decode_dev(out, slot, [n], 1, J.default_frame(W, H), back, status, stream=st.cuda_stream)
    torch.cuda.synchronize()
    assert int(status.item()) == 0 and bool((back == coefs).all())
    raw = np.frombuffer(single, dtype=np.uint8)
    ff = int((raw == 0xFF).sum())
    assert n == (int(nb[1].item()) + 7) // 8 + ff and bool((raw[np.nonzero(raw[:-1] == 0xFF)[0] + 1] == 0).all())
    # (3) libjpeg (Pillow) reads our file and lands near the source image
    PIL = pytest.importorskip("PIL.Image")
    W2, H2 = 3840, 2160
    d2 = synth_dev(ctx, W2, H2)
    r, g, b = (d2[c].cpu().numpy() for c in range(3))
    scan, _ = ctx.encode(r, g, b, W2, H2)
    # the reference's header bytes, written by the host mirror (include/jpezy/jpezy_writer.hpp) -- here through the CLI-free path:
    import oracle as orc
    f = orc.Oracle().header(W2, H2) + scan + b"\xff\xd9"
    im = np.asarray(PIL.open(io.BytesIO(f)).convert("RGB")).astype(np.float64)
    src = np.stack([r, g, b], -1).astype(np.float64)
    psnr = 10 * np.log10(255.0 ** 2 / ((im - src) ** 2).mean())
    assert psnr > 30.0, psnr


def test_c3_batch_equals_per_frame(ctx):
    W, H, N = 1920, 1080, 6
    d = torch.empty((3, N, H, W), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.synth_dev(d[0], d[1], d[2], W, H, N, 100, 0)
    torch.cuda.synchronize()
    slot = W * H
    out = torch.zeros((N, slot), dtype=torch.uint8, device="cuda")
    nb = torch.zeros(N, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.encode_batch_dev(d[0], d[1], d[2], W, H, N, False, out, slot, nb, None)
    torch.cuda.synchronize()
    h = d.cpu().numpy()
    frame = J.default_frame(W, H)
    pl = capi.plane_bytes(frame)
    planes = torch.zeros((3, N, pl), dtype=torch.uint8, device="cuda")
    status = torch.zeros(N, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.decode_batch_dev(out, slot, nb.cpu().numpy(), N, frame, False, planes[0], planes[1], planes[2], pl, status)
    torch.cuda.synchronize()
    assert not status.any()
    ph = planes.cpu().numpy()
    for k in range(N):
        scan, _ = ctx.encode(h[0, k], h[1, k], h[2, k], W, H)
        assert out[k, : int(nb[k])].cpu().numpy().tobytes() == scan
        if k < 2:
            R, G, B = ctx.decode(scan, frame)
            assert (ph[0, k] == R).all() and (ph[1, k] == G).all() and (ph[2, k] == B).all()
