"""-m gpu parity tests of the encoder path (C ABI -> CUDA kernels) against the CPU oracle.

Bars (BASELINE.json north_star): quantised coefficients bit-exact (the exact-order recompute path
makes even the boundary cases agree, so the test demands 0 mismatches and reports the guard count);
given identical coefficients the entropy-coded segment is byte-identical; whole file byte-identical.
"""
import numpy as np
import pytest
import torch

import jpezy_b200 as J
from jpezy_b200 import capi
from gpu_util import gpu_coefs, gpu_entropy, planes, to_dev

pytestmark = pytest.mark.gpu

SIZES = [(64, 48), (200, 120), (1, 1), (17, 33), (16, 16), (250, 7), (512, 512)]


def test_library_is_the_cuda_path(ctx):
    # the product path must be the in-tree CUDA library, never a CPU stand-in
    assert capi.load_library()._name.endswith("jpezy_b200/libjpezy_b200.so")
    assert ctx.stat(capi.STAT_KERNEL_LAUNCHES) >= 0


@pytest.mark.parametrize("family", [0, 1, 2])
def test_synth_device_matches_numpy(ctx, family):
    W, H = 200, 72
    d = torch.empty((3, 2, H, W), dtype=torch.uint8, device="cuda")
    ctx.synth_dev(d[0], d[1], d[2], W, H, nimg=2, first_frame=5, family=family, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    h = d.cpu().numpy()
    for f in range(2):
        r, g, b = J.synth.image(family, W, H, frame=5 + f)
        assert (h[0, f] == r).all() and (h[1, f] == g).all() and (h[2, f] == b).all()


@pytest.mark.parametrize("W,H", SIZES)
@pytest.mark.parametrize("family", [0, 1, 2])
@pytest.mark.parametrize("gray", [False, True])
def test_coefficients_bit_exact(ctx, oracle, W, H, family, gray):
    r, g, b = planes(family, W, H)
    want = oracle.coefs(r, g, b, W, H, gray=gray)
    got = gpu_coefs(ctx, r, g, b, W, H, gray=gray)[0]
    bad = np.argwhere(want != got)
    assert bad.shape[0] == 0, "first mismatches (mcu, block, zz): %s want %s got %s" % (
        bad[:5].tolist(), want[tuple(bad[:5].T)].tolist(), got[tuple(bad[:5].T)].tolist())


@pytest.mark.parametrize("W,H", [(64, 48), (208, 128), (512, 512), (1920, 16), (4080, 48), (1024, 272)])
@pytest.mark.parametrize("family", [0, 1, 2])
@pytest.mark.parametrize("gray", [False, True])
def test_forward_kernel_16_byte_row_loads_bit_exact(ctx, oracle, W, H, family, gray):
    """widths that are multiples of 16 take the 16-byte row loads of the production forward kernel: coefficients and scan
    bit-exact on whole and partial 32-MCU tiles and on frames of one MCU row (1920x16)."""
    r, g, b = planes(family, W, H)
    want = oracle.coefs(r, g, b, W, H, gray=gray)
    got = gpu_coefs(ctx, r, g, b, W, H, gray=gray)[0]
    scan, _ = ctx.encode(r, g, b, W, H, gray=gray)
    assert (want == got).all(), "%d coefficients differ" % int((want != got).sum())
    assert scan == oracle.encode(r, g, b, W, H, gray=gray, scan_only=True)


def test_guard_path_is_exercised(ctx, oracle):
    # flat gray tiles: every DC sits on a multiple of its quantiser whenever 8p % 16 == 0 -> the reference's FP64
    # rounding decides (SURVEY.md 7, hard part 1: DC = 8p -+ 1 ulp); the DC path evaluates ((S*c)*c)/4 as the reference does
    W, H = 256, 64
    r, g, b = planes(2, W, H)
    assert (gpu_coefs(ctx, r, g, b, W, H)[0] == oracle.coefs(r, g, b, W, H)).all()
    # an AC coefficient exactly on a boundary: columns a,b,b,a,a,b,b,a give F(0,4) = 4(a-b); 4*6 = 24 = q(0,4)
    found = False
    for base in range(20, 200, 7):
        row = np.array([base + 6, base, base, base + 6, base + 6, base, base, base + 6] * 4, dtype=np.uint8)
        v = np.tile(row, (16, 1))
        c, raw = oracle.coefs(v, v, v, 32, 16, want_raw=True)
        if abs(abs(raw[0, 0, 4]) - 24.0) < 1e-9:
            found = True
            before = ctx.stat(capi.STAT_GUARD_FWD)
            assert (gpu_coefs(ctx, v, v, v, 32, 16)[0] == c).all()
            assert ctx.stat(capi.STAT_GUARD_FWD) > before, "tier-3 (exact operation order) path was not taken"
            break
    assert found


def test_exhaustive_colour_conversion(ctx, oracle):
    """every (r, g, b) triple exactly once: a 4096 x 4096 image holds all 2^24 colours.  All of its coefficients must equal the
    oracle's -- luma sees every triple; the triple of pixel (x, y) is arranged so that the even/even positions, the only ones
    chroma is taken from (decimation, src/encoder/jpezy_encoder.hpp:116-143), run through every triple as well over the four
    images of the sweep (the (x, y) -> index map is shifted by (0|1, 0|1))."""
    W = H = 4096
    yy, xx = np.meshgrid(np.arange(H, dtype=np.uint32), np.arange(W, dtype=np.uint32), indexing="ij")
    for dy in (0, 1):
        for dx in (0, 1):
            idx = (((yy + dy) % H) * W + ((xx + dx) % W)).astype(np.uint32)
            # a permutation of the index that spreads neighbouring triples (otherwise every block is a smooth ramp)
            idx = (idx * np.uint32(2654435761)) & np.uint32(0xffffff)
            r = (idx & 255).astype(np.uint8)
            g = ((idx >> 8) & 255).astype(np.uint8)
            b = ((idx >> 16) & 255).astype(np.uint8)
            if dy == 0 and dx == 0:
                key = (r.astype(np.uint32) | (g.astype(np.uint32) << 8) | (b.astype(np.uint32) << 16)).ravel()
                assert np.unique(key).size == 1 << 24, "the sweep image must hold every colour"
            got = gpu_coefs(ctx, r, g, b, W, H)[0]
            want = oracle.coefs(r, g, b, W, H)
            nd = int((got != want).sum())
            assert nd == 0, "%d coefficients differ (shift %d,%d)" % (nd, dx, dy)


def test_gray_pixels_colour_boundaries(ctx, oracle):
    # r=g=b=v: the exact Y is the integer v-128, so the FP64 rounding of the reference decides 30 of 256 values
    W, H = 256, 16
    v = np.tile(np.arange(256, dtype=np.uint8), (H, 1))
    assert (gpu_coefs(ctx, v, v, v, W, H)[0] == oracle.coefs(v, v, v, W, H)).all()


@pytest.mark.parametrize("W,H", SIZES)
@pytest.mark.parametrize("family", [0, 1, 2])
def test_entropy_segment_byte_identical_given_coefficients(ctx, oracle, W, H, family):
    r, g, b = planes(family, W, H)
    coefs = oracle.coefs(r, g, b, W, H)
    want = oracle.scan_from_coefs(coefs)
    got, nbits = gpu_entropy(ctx, coefs, W, H)
    assert got[0] == want
    assert (nbits[0] + 7) // 8 <= len(want)


def test_entropy_extreme_coefficients(ctx, oracle):
    # runs >= 16 (ZRL), coefficient 63 non-zero (no EOB), max magnitudes, 0xFF-heavy output
    rng = np.random.default_rng(3)
    n = 24
    c = np.zeros((n, 6, 64), dtype=np.int16)
    c[0, 0, 63] = 1                      # run of 62 -> 3 ZRL, no EOB
    c[1, :, 0] = [1023, -1023, 512, -512, 255, -255]
    c[2, 1, 17] = -3; c[2, 1, 50] = 7
    c[3] = rng.integers(-1023, 1024, size=(6, 64))
    c[4:] = (rng.integers(-40, 41, size=(n - 4, 6, 64)) * (rng.random((n - 4, 6, 64)) < 0.15)).astype(np.int16)
    W, H = 16 * n, 16
    want = oracle.scan_from_coefs(c)
    got, _ = gpu_entropy(ctx, c, W, H)
    assert got[0] == want
    assert b"\xff\x00" in want


@pytest.mark.parametrize("where", ["dc", "ac"])
def test_entropy_refuses_coefficients_without_a_code(ctx, where):
    """a DC difference of more than 11 bits or an AC value of more than 10 bits has no code in the Annex K tables: the reference
    throws (src/encoder/jpezy_encoder.hpp:186,207); the device path must report the image (byte count < 0 = UINT64_MAX) instead
    of emitting a stream with missing symbols -- and must leave the other image of the batch alone"""
    n = 4
    c = np.zeros((2, n, 6, 64), dtype=np.int16)
    c[:, :, :, 0] = 5
    if where == "dc":
        c[1, 2, 0, 0] = 32000                      # difference to the previous block: 15 bits
    else:
        c[1, 1, 3, 9] = -2000                      # 11 bits
    W, H = 16 * n, 16
    got, _ = gpu_entropy(ctx, c, W, H, nimg=2)
    assert got[0] is not None and len(got[0]) > 0
    assert got[1] is None


@pytest.mark.parametrize("pad_ones", [1, 0])
def test_pad_policy(ctx, oracle, pad_ones):
    W, H = 40, 24
    r, g, b = planes(0, W, H)
    coefs = oracle.coefs(r, g, b, W, H)
    ctx.set_option(capi.OPT_PAD_ONES, pad_ones)
    try:
        got, _ = gpu_entropy(ctx, coefs, W, H)
    finally:
        ctx.set_option(capi.OPT_PAD_ONES, 1)
    assert got[0] == oracle.scan_from_coefs(coefs, pad_ones=bool(pad_ones))


@pytest.mark.parametrize("value", [2, 3, -1])
def test_transform_option_takes_only_production_or_validation(ctx, value):
    with pytest.raises(capi.JpezyError) as e:
        ctx.set_option(capi.OPT_TRANSFORM, value)
    assert e.value.code == capi.EINVAL
    for ok in (1, 0):
        ctx.set_option(capi.OPT_TRANSFORM, ok)


@pytest.mark.parametrize("W,H,family,gray", [(200, 120, 0, False), (512, 512, 0, False), (512, 512, 1, False), (96, 80, 2, True),
                                             (333, 77, 1, True)])
def test_host_encode_file_byte_identical(ctx, oracle, W, H, family, gray):
    r, g, b = planes(family, W, H)
    want = oracle.encode(r, g, b, W, H, gray=gray)
    scan, nbits = ctx.encode(r, g, b, W, H, gray=gray)
    got = oracle.header(W, H, gray=gray) + scan + b"\xff\xd9"
    assert got == want


def test_batch_encode_matches_single(ctx, oracle):
    W, H, N = 136, 72, 5
    imgs = [planes(f % 2, W, H, frame=f) for f in range(N)]
    R = to_dev(np.stack([i[0] for i in imgs])); G = to_dev(np.stack([i[1] for i in imgs])); B = to_dev(np.stack([i[2] for i in imgs]))
    slot = W * H * 3
    out = torch.zeros((N, slot), dtype=torch.uint8, device="cuda")
    nbytes = torch.zeros(N, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()      # torch's stream and the context's own (non-blocking) stream are not ordered with each other
    ctx.encode_batch_dev(R, G, B, W, H, N, False, out, slot, nbytes, None, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    o, nb = out.cpu().numpy(), nbytes.cpu().numpy()
    for f in range(N):
        assert o[f, : nb[f]].tobytes() == oracle.encode(*imgs[f], W, H, scan_only=True)


def test_capacity_error(ctx):
    W, H = 128, 128
    r, g, b = planes(1, W, H)
    with pytest.raises(J.JpezyError) as e:
        ctx.encode(r, g, b, W, H, scan_cap=64)
    assert e.value.code == capi.ECAPACITY


def test_invalid_arguments(ctx):
    with pytest.raises(J.JpezyError) as e:
        ctx.transform_fwd_dev(1, 1, 1, 0, 10, 1, False, 1)
    assert e.value.code == capi.EINVAL
    with pytest.raises(J.JpezyError):
        ctx.transform_fwd_dev(1, 1, 1, 70000, 10, 1, False, 1)
