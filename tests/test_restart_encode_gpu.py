"""-m gpu tests of restart intervals in the encoders (JPEZYB200_OPT_RESTART_INTERVAL): every single-context encode path writes
the oracle's segment of each interval (predictors from 0, padded to a byte) joined by RST0..RST7 in cyclic order, the
optimised tables are fitted to the restart stream's symbols, and the files decode like the restart-less ones in the oracle,
in Pillow (libjpeg), in the library's own decoder and through the CLIs.

The module has a context of its own; the session context keeps interval 0."""
import ctypes as C
import io
import os
import subprocess

import numpy as np
import pytest
import torch

import jpezy_b200 as J
from jpezy_b200 import capi
from jpezy_b200.capi import EINVAL, EUNSUPPORTED, ECAPACITY, OPT_PAD_ONES, OPT_RESTART_INTERVAL, _dp
from gpu_util import planes, to_dev
from jpeg_build import bit_length, symbol_hist
from test_huffopt_gpu import check_table, with_tables

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "jpezy_b200", "bin")
HB = capi.HUFF_TABLES_BYTES
SIZES = [(8, 8), (17, 33), (200, 120), (1920, 1080)]


@pytest.fixture(scope="module")
def rctx():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    torch.cuda.init()
    c = J.Context(0)
    yield c
    c.close()


class interval:
    """the context's restart interval (and pad bits) for the duration of a with-block"""

    def __init__(self, ctx, mcus, pad_ones=1):
        self.ctx, self.mcus, self.pad = ctx, mcus, pad_ones

    def __enter__(self):
        self.ctx.set_option(OPT_RESTART_INTERVAL, self.mcus)
        self.ctx.set_option(OPT_PAD_ONES, self.pad)

    def __exit__(self, *exc):
        self.ctx.set_option(OPT_RESTART_INTERVAL, 0)
        self.ctx.set_option(OPT_PAD_ONES, 1)


def intervals_of(W, H):
    n = capi.num_mcus(W, H)
    return sorted({1, 2, 7, (W + 15) // 16, max(n - 1, 1), n, 65535})


# ---- the expected segment ----------------------------------------------------------------------------------------------
def oracle_scan(oracle, coefs, pad_ones=True):
    """-> (segment, Huffman bits) of one restart-less stream whose predictors start at 0"""
    c = np.ascontiguousarray(coefs, dtype=np.int16).reshape(-1, 6, 64)
    cap = c.size * 4 + 1024
    out = np.zeros(cap, np.uint8)
    n, nb = C.c_size_t(0), C.c_uint64(0)
    assert oracle.lib.orc_scan_from_coefs(c.ctypes.data_as(C.POINTER(C.c_int16)), c.shape[0], int(pad_ones),
                                          out.ctypes.data_as(C.POINTER(C.c_uint8)), cap, C.byref(n), C.byref(nb)) == 0
    return out[: n.value].tobytes(), nb.value


def restart_scan(oracle, coefs, R, pad_ones=True):
    """the oracle's segment of every interval of R MCUs, joined by RSTn markers -> (segment, Huffman bits)"""
    c = np.asarray(coefs).reshape(-1, 6, 64)
    parts, bits = bytearray(), 0
    for i, m0 in enumerate(range(0, c.shape[0], R)):
        s, nb = oracle_scan(oracle, c[m0:m0 + R], pad_ones)
        if i:
            parts += bytes([0xFF, 0xD0 + (i - 1) % 8])
        parts += s
        bits += nb
    return bytes(parts), bits


def rst_symbol_hist(coefs, R):
    """symbol_hist of the restart stream: the DC predictors restart at 0 in every interval of R MCUs"""
    c = np.asarray(coefs, dtype=np.int64).reshape(-1, 6, 64)
    hist, extra = symbol_hist(c)
    dc = c[:, :, 0]
    start = (np.arange(c.shape[0]) % R) == 0
    for cls, seq, first in ((0, dc[:, :4].reshape(-1), np.repeat(start, 4) & (np.arange(4 * c.shape[0]) % 4 == 0)),
                            (1, dc[:, 4], start), (1, dc[:, 5], start)):
        old = np.minimum(bit_length(np.diff(seq, prepend=0)), 11)
        pred = np.concatenate([[0], seq[:-1]])
        pred[first] = 0
        new = np.minimum(bit_length(seq - pred), 11)
        hist[cls, :16] += np.bincount(new, minlength=16) - np.bincount(old, minlength=16)
        extra += int(new.sum()) - int(old.sum())
    return hist, extra


def check_rst_tables(ht, coefs, R):
    """the four tables fitted to the restart stream -> the un-stuffed bit count they give"""
    hist, total = rst_symbol_hist(coefs, R)
    for cls in (0, 1):
        dcl = check_table(ht[0][cls], hist[cls, :16])
        acl = check_table(ht[1][cls], hist[cls, 16:])
        total += sum(int(hist[cls, s]) * L for s, L in dcl.items()) + sum(int(hist[cls, 16 + s]) * L for s, L in acl.items())
    return total


def with_dri(header, R):
    """the header with a DRI segment in front of SOS"""
    i = header.rindex(b"\xff\xda")
    return header[:i] + bytes([0xFF, 0xDD, 0, 4, R >> 8, R & 0xFF]) + header[i:]


# ---- device helpers -------------------------------------------------------------------------------------------------------
def dev_entropy(ctx, coefs, W, H, nimg=1, slot=None, optimized=False):
    dc = to_dev(np.ascontiguousarray(coefs, dtype=np.int16))
    slot = int(slot or max(W * H * 3, 10240))
    out = torch.zeros((nimg, slot), dtype=torch.uint8, device="cuda")
    nbytes = torch.zeros(nimg, dtype=torch.int64, device="cuda")
    nbits = torch.zeros(nimg, dtype=torch.int64, device="cuda")
    d_ht = torch.zeros(nimg * HB, dtype=torch.uint8, device="cuda")
    sp = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    if optimized:
        ctx.entropy_encode_optimized_dev(dc, W, H, nimg, False, out, slot, d_ht, nbytes, nbits, stream=sp)
    else:
        ctx.entropy_encode_dev(dc, W, H, nimg, False, out, slot, nbytes, nbits, stream=sp)
    torch.cuda.synchronize()
    nb, o, h = nbytes.cpu().numpy(), out.cpu().numpy(), d_ht.cpu().numpy()
    scans = [o[i, : nb[i]].tobytes() if nb[i] >= 0 else None for i in range(nimg)]
    return scans, nbits.cpu().numpy(), [J.huff_tables(h[i * HB:(i + 1) * HB]) for i in range(nimg)]


def dev_batch(ctx, imgs, W, H, gray=False, optimized=False):
    n = len(imgs)
    d_in = to_dev(np.stack([np.stack(p) for p in imgs], 1))   # [3][n][H][W]
    slot = max(W * H * 3, 10240)
    out = torch.zeros((n, slot), dtype=torch.uint8, device="cuda")
    nbytes = torch.zeros(n, dtype=torch.int64, device="cuda")
    nbits = torch.zeros(n, dtype=torch.int64, device="cuda")
    d_ht = torch.zeros(n * HB, dtype=torch.uint8, device="cuda")
    sp = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    if optimized:
        ctx.encode_batch_optimized_dev(d_in[0], d_in[1], d_in[2], W, H, n, gray, out, slot, d_ht, nbytes, nbits, stream=sp)
    else:
        ctx.encode_batch_dev(d_in[0], d_in[1], d_in[2], W, H, n, gray, out, slot, nbytes, nbits, stream=sp)
    torch.cuda.synchronize()
    nb, o, h = nbytes.cpu().numpy(), out.cpu().numpy(), d_ht.cpu().numpy()
    return ([o[i, : nb[i]].tobytes() for i in range(n)], nbits.cpu().numpy(),
            [J.huff_tables(h[i * HB:(i + 1) * HB]) for i in range(n)])


_COEFS = {}


def coefs_of(oracle, family, W, H, gray):
    key = (family, W, H, gray)
    if key not in _COEFS:
        r, g, b = planes(family, W, H)
        _COEFS[key] = oracle.coefs(r, g, b, W, H, gray=gray)
    return _COEFS[key]


# ---- byte-exact against the oracle ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,H", SIZES)
@pytest.mark.parametrize("family", [0, 1, 2])
@pytest.mark.parametrize("gray", [False, True])
def test_segment_matches_oracle(rctx, oracle, W, H, family, gray):
    coefs = coefs_of(oracle, family, W, H, gray)
    for R in intervals_of(W, H):
        for pad in (1, 0):
            want, bits = restart_scan(oracle, coefs, R, pad_ones=bool(pad))
            with interval(rctx, R, pad):
                scans, nbits, _ = dev_entropy(rctx, coefs, W, H)
            assert scans[0] == want, (R, pad)
            assert nbits[0] == bits, (R, pad)


# ---- every entry point -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,H", [(200, 120), (1920, 1080)])
@pytest.mark.parametrize("family", [0, 1])
@pytest.mark.parametrize("gray", [False, True])
def test_entry_points_agree(rctx, oracle, W, H, family, gray):
    r, g, b = planes(family, W, H)
    coefs = oracle.coefs(r, g, b, W, H, gray=gray)
    for R in (1, 5, (W + 15) // 16):
        want, bits = restart_scan(oracle, coefs, R)
        with interval(rctx, R):
            host, host_bits = rctx.encode(r, g, b, W, H, gray=gray)
            ent, ent_bits, _ = dev_entropy(rctx, coefs, W, H)
            bat, bat_bits, _ = dev_batch(rctx, [(r, g, b)], W, H, gray=gray)
        assert host == ent[0] == bat[0] == want
        assert host_bits == ent_bits[0] == bat_bits[0] == bits


def test_host_batch_equals_single_calls(rctx):
    W, H, n = 200, 120, 9
    imgs = [planes(i % 3, W, H, frame=i) for i in range(n)]
    slot = W * H * 3
    r, g, b = (np.ascontiguousarray(np.stack([im[c].reshape(-1) for im in imgs])) for c in range(3))
    out = np.zeros(n * slot, np.uint8)
    nb = np.zeros(n, np.uint64)
    try:
        rctx.set_option(capi.OPT_BATCH_GROUP_BYTES, 3 * W * H * 2)   # two images per group: five groups
        with interval(rctx, 3):
            rctx.encode_batch(r, g, b, W, H, n, False, out, slot, nb)
            single = [rctx.encode(*im, W, H)[0] for im in imgs]
    finally:
        rctx.set_option(capi.OPT_BATCH_GROUP_BYTES, 96 << 20)
    assert [out[i * slot: i * slot + int(nb[i])].tobytes() for i in range(n)] == single


@pytest.mark.parametrize("W,H", [(17, 33), (200, 120), (1920, 1080)])
@pytest.mark.parametrize("family", [0, 1, 2])
@pytest.mark.parametrize("gray", [False, True])
def test_optimized_tables_fit_restart_stream(rctx, oracle, W, H, family, gray):
    r, g, b = planes(family, W, H)
    coefs = oracle.coefs(r, g, b, W, H, gray=gray)
    for R in (1, 4, (W + 15) // 16):
        with interval(rctx, R):
            scan, nbits, ht = rctx.encode_optimized(r, g, b, W, H, gray=gray)
            ent, ent_bits, ent_ht = dev_entropy(rctx, coefs, W, H, optimized=True)
            bat, bat_bits, bat_ht = dev_batch(rctx, [(r, g, b)], W, H, gray=gray, optimized=True)
        assert nbits == check_rst_tables(ht, coefs, R)
        assert scan == ent[0] == bat[0] and nbits == ent_bits[0] == bat_bits[0]
        assert bytes(ht) == bytes(ent_ht[0]) == bytes(bat_ht[0])
        f = with_dri(with_tables(oracle.header(W, H, gray=gray), ht), R) + scan + b"\xff\xd9"
        assert (oracle.decode_coefs(f) == coefs).all()


# ---- independent decoders ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,H", [(17, 33), (200, 120), (1920, 1080)])
@pytest.mark.parametrize("family", [0, 1, 2])
@pytest.mark.parametrize("gray", [False, True])
def test_files_decode_like_restart_less_files(rctx, oracle, W, H, family, gray):
    from PIL import Image
    r, g, b = planes(family, W, H)
    coefs = oracle.coefs(r, g, b, W, H, gray=gray)
    header = oracle.header(W, H, gray=gray)
    ref = oracle.encode(r, g, b, W, H, gray=gray)
    px_k = np.asarray(Image.open(io.BytesIO(ref)))
    scan_o, _, ht_o = rctx.encode_optimized(r, g, b, W, H, gray=gray)
    px_o = np.asarray(Image.open(io.BytesIO(with_tables(header, ht_o) + scan_o + b"\xff\xd9")))
    for R in (1, 3, (W + 15) // 16):
        with interval(rctx, R):
            scan, _ = rctx.encode(r, g, b, W, H, gray=gray)
            scan2, _, ht = rctx.encode_optimized(r, g, b, W, H, gray=gray)
        f = with_dri(header, R) + scan + b"\xff\xd9"
        assert (oracle.decode_coefs(f) == coefs).all()
        assert (np.asarray(Image.open(io.BytesIO(f))) == px_k).all()
        f2 = with_dri(with_tables(header, ht), R) + scan2 + b"\xff\xd9"
        assert (np.asarray(Image.open(io.BytesIO(f2))) == px_o).all()


@pytest.mark.parametrize("W,H", [(200, 120), (3840, 2160)])
@pytest.mark.parametrize("gray", [False, True])
def test_library_decoder_reads_restart_streams(rctx, W, H, gray):
    n = 2
    imgs = [planes(i, W, H, frame=i) for i in range(n)]
    want = [rctx.decode(rctx.encode(*im, W, H, gray=gray)[0], J.default_frame(W, H), gray=gray) for im in imgs]
    frame = J.default_frame(W, H)
    need = capi.plane_bytes(frame)
    for R in (1, 8, (W + 15) // 16):
        frame.restart_interval = R
        with interval(rctx, R):
            host = [rctx.decode(rctx.encode(*im, W, H, gray=gray)[0], frame, gray=gray) for im in imgs]
            scans, _, _ = dev_batch(rctx, imgs, W, H, gray=gray)
        for got, exp in zip(host, want):
            assert all((x == y).all() for x, y in zip(got, exp)), R
        # device resident: the encoder's lengths stay on the device
        slot = max(len(s) for s in scans) + 64
        d_scan = torch.zeros((n, slot), dtype=torch.uint8, device="cuda")
        for i, s in enumerate(scans):
            d_scan[i, : len(s)] = torch.frombuffer(bytearray(s), dtype=torch.uint8)
        d_len = torch.tensor([len(s) for s in scans], dtype=torch.int64, device="cuda")
        outs = [torch.zeros(n * need, dtype=torch.uint8, device="cuda") for _ in range(3)]
        st = torch.zeros(n, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        rctx.decode_batch_dev2(d_scan, slot, d_len, slot, n, frame, gray, *outs, need, st, stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert (st.cpu().numpy() == 0).all()
        o = [x.cpu().numpy().reshape(n, need) for x in outs]
        for i in range(n):
            assert all((o[c][i] == want[i][c]).all() for c in range(3)), R


# ---- errors ---------------------------------------------------------------------------------------------------------------------
def test_option_range(rctx):
    for bad in (-1, 65536, 1 << 40):
        with pytest.raises(J.JpezyError) as e:
            rctx.set_option(OPT_RESTART_INTERVAL, bad)
        assert e.value.code == EINVAL
    for ok in (0, 1, 65535):
        rctx.set_option(OPT_RESTART_INTERVAL, ok)
    rctx.set_option(OPT_RESTART_INTERVAL, 0)


def test_sharded_and_group_encoders_refuse_intervals(rctx):
    W, H = 64, 64
    r, g, b = (to_dev(p) for p in planes(0, W, H))
    last = torch.zeros(4, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    with interval(rctx, 2):
        with pytest.raises(J.JpezyError) as e:
            rctx.shard_encode_a(r, g, b, W, H, 0, 4, 0, False, last)
        assert e.value.code == EUNSUPPORTED
    rctx.shard_encode_a(r, g, b, W, H, 0, 4, 0, False, last)   # and works again at 0
    torch.cuda.synchronize()

    L = rctx.lib
    L.jpezyb200_group_create.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_void_p)]
    L.jpezyb200_group_ctx.argtypes = [C.c_void_p, C.c_uint32]
    L.jpezyb200_group_ctx.restype = C.c_void_p
    L.jpezyb200_group_destroy.argtypes = [C.c_void_p]
    L.jpezyb200_group_destroy.restype = None
    L.jpezyb200_group_encode.argtypes = [C.c_void_p] + [C.POINTER(C.c_void_p)] * 3 + [C.c_uint32, C.c_uint32, C.c_int, C.c_void_p,
                                                                                       C.c_size_t, C.POINTER(C.c_uint64)]
    grp = C.c_void_p()
    assert L.jpezyb200_group_create(1, (C.c_int * 1)(0), C.byref(grp)) == 0
    try:
        gctx = L.jpezyb200_group_ctx(grp, 0)
        assert L.jpezyb200_set_option(gctx, OPT_RESTART_INTERVAL, 4) == 0
        dst = torch.zeros(W * H * 3, dtype=torch.uint8, device="cuda")
        nb = C.c_uint64(0)
        ptrs = [(C.c_void_p * 1)(_dp(x)) for x in (r, g, b)]
        assert L.jpezyb200_group_encode(grp, *ptrs, W, H, 0, _dp(dst), W * H * 3, C.byref(nb)) == EUNSUPPORTED
        assert L.jpezyb200_set_option(gctx, OPT_RESTART_INTERVAL, 0) == 0
        assert L.jpezyb200_group_encode(grp, *ptrs, W, H, 0, _dp(dst), W * H * 3, C.byref(nb)) == 0
    finally:
        L.jpezyb200_group_destroy(grp)


def test_slot_too_small_for_the_markers(rctx, oracle):
    W, H = 200, 120
    r, g, b = planes(0, W, H)
    coefs = oracle.coefs(r, g, b, W, H)
    plain, _ = oracle_scan(oracle, coefs)
    want, _ = restart_scan(oracle, coefs, 1)
    assert len(plain) < len(want)
    slot = len(want) - 1
    assert dev_entropy(rctx, coefs, W, H, slot=slot)[0][0] == plain   # the restart-less segment fits
    with interval(rctx, 1):
        scans, _, _ = dev_entropy(rctx, coefs, W, H, slot=slot)
        assert scans[0] is None
        assert dev_entropy(rctx, coefs, W, H, slot=len(want))[0][0] == want
        with pytest.raises(J.JpezyError) as e:
            rctx.encode(r, g, b, W, H, scan_cap=slot)
        assert e.value.code == ECAPACITY


def test_coefficient_without_code_reports_overflow(rctx):
    W, H = 32, 16
    coefs = np.zeros((2, 6, 64), np.int16)
    coefs[1, 2, 5] = 1024   # an 11-bit AC value
    with interval(rctx, 1):
        for opt in (False, True):
            scans, nbits, _ = dev_entropy(rctx, coefs, W, H, optimized=opt)
            assert scans[0] is None and nbits[0] == -1


def test_interval_zero_again_equals_fresh_context(rctx):
    W, H = 200, 120
    imgs = [planes(f, W, H) for f in range(3)]
    with interval(rctx, 2):
        for im in imgs:
            rctx.encode(*im, W, H)
            rctx.encode_optimized(*im, W, H)
    fresh = J.Context(0)
    try:
        for im in imgs:
            assert rctx.encode(*im, W, H) == fresh.encode(*im, W, H)
            a, b = rctx.encode_optimized(*im, W, H), fresh.encode_optimized(*im, W, H)
            assert a[:2] == b[:2] and bytes(a[2]) == bytes(b[2])
            assert dev_batch(rctx, [im], W, H)[0] == dev_batch(fresh, [im], W, H)[0]
    finally:
        fresh.close()


# ---- CLI -------------------------------------------------------------------------------------------------------------------------
def write_ppm(path, r, g, b):
    H, W = r.shape
    rgb = np.stack([r, g, b], -1).reshape(-1, 3)
    path.write_text("P3\n%d %d\n255\n" % (W, H) + "\n".join("%d %d %d" % tuple(p) for p in rgb) + "\n")


def markers(f):
    """(DRI value or None, the RSTn marker bytes in order) of a JPEG file"""
    i, dri = 2, None
    while f[i + 1] != 0xDA:
        ln = (f[i + 2] << 8) | f[i + 3]
        if f[i + 1] == 0xDD:
            assert dri is None, "more than one DRI"
            dri = (f[i + 4] << 8) | f[i + 5]
        i += 2 + ln
    i += 2 + ((f[i + 2] << 8) | f[i + 3])
    rst = [f[k + 1] for k in range(i, len(f) - 1) if f[k] == 0xFF and 0xD0 <= f[k + 1] <= 0xD7]
    return dri, rst


@pytest.mark.parametrize("flags,mcus", [(["--restart", "2"], lambda hu: 2 * hu), (["--restart", "5B"], lambda hu: 5),
                                        (["--optimize", "--restart", "1"], lambda hu: hu),
                                        (["--restart", "3B", "--optimize"], lambda hu: 3),
                                        (["--gray", "--restart", "1B"], lambda hu: 1),
                                        (["--restart", "1", "--gray", "--optimize"], lambda hu: hu),
                                        (["--optimize", "--gray", "--restart", "7b"], lambda hu: 7),
                                        (["--restart", "0"], lambda hu: 0)])
def test_cli_restart(tmp_path, oracle, flags, mcus):
    from PIL import Image
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "jpezy_b200", "cli"), "-s"])
    enc, dec = os.path.join(BIN, "jpezy_encode"), os.path.join(BIN, "jpezy_decode")
    W, H = 129, 65
    r, g, b = planes(1, W, H)
    src = tmp_path / "in.ppm"
    write_ppm(src, r, g, b)
    gray = "--gray" in flags
    base = [f for f in flags if f in ("--optimize", "--gray")]
    for name, extra in (("plain", base), ("rst", flags)):
        p = subprocess.run([enc, str(src), str(tmp_path / (name + ".jpg")), *extra], capture_output=True, text=True)
        assert p.returncode == 0, p.stderr
        q = subprocess.run([dec, str(tmp_path / (name + ".jpg")), str(tmp_path / (name + ".ppm")), *(["--gray"] if gray else [])],
                           capture_output=True, text=True)
        assert q.returncode == 0, q.stderr
    fp, fr = (tmp_path / "plain.jpg").read_bytes(), (tmp_path / "rst.jpg").read_bytes()
    R = mcus((W + 15) // 16)
    nint = -(-capi.num_mcus(W, H) // R) if R else 1
    dri, rst = markers(fr)
    assert dri == (R or None)
    assert rst == [0xD0 + i % 8 for i in range(nint - 1)]
    if not R:
        assert fr == fp
    assert (oracle.decode_coefs(fr) == oracle.coefs(r, g, b, W, H, gray=gray)).all()
    assert (tmp_path / "rst.ppm").read_text() == (tmp_path / "plain.ppm").read_text()
    assert (np.asarray(Image.open(io.BytesIO(fr))) == np.asarray(Image.open(io.BytesIO(fp)))).all()


@pytest.mark.parametrize("bad", [["--restart"], ["--restart", "x"], ["--restart", "-1"], ["--restart", "65536B"],
                                 ["--restart", "10000"], ["--restart", "2", "--restart", "3"], ["--restart", "B"]])
def test_cli_restart_bad_values(tmp_path, bad):
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "jpezy_b200", "cli"), "-s"])
    W, H = 129, 65
    src = tmp_path / "in.ppm"
    write_ppm(src, *planes(0, W, H))
    p = subprocess.run([os.path.join(BIN, "jpezy_encode"), str(src), str(tmp_path / "o.jpg"), *bad], capture_output=True, text=True)
    assert p.returncode == 1 and "Usage: jpezy_encode" in p.stderr
