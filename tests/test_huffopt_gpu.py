"""-m gpu tests of the optimised Huffman tables (jpezyb200_*_optimized*): the device tables equal a Python restatement of
T.81 section K.2 written after libjpeg's jpeg_gen_optimal_table, fed with the symbol counts of the oracle's coefficients;
the segments decode to the same coefficients and pixels as the Annex K files, and are never longer."""
import io
import os
import subprocess

import numpy as np
import pytest
import torch

import jpezy_b200 as J
from jpezy_b200 import capi
from gpu_util import planes, to_dev
from jpeg_build import dht, fibonacci_coefs, gen_optimal_table, symbol_hist

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "jpezy_b200", "bin")
TABLE_SIZES = [(1, 1), (17, 33), (200, 120), (512, 512), (1920, 1080)]
HB = capi.HUFF_TABLES_BYTES


# ---- Python reference ------------------------------------------------------------------------------
def code_lengths(bits, huffval):
    return {s: L for s, L in zip(huffval, [L for L in range(1, 17) for _ in range(bits[L - 1])])}


def check_table(h, counts):
    """device record == reference; at most 16-bit codes, Kraft, no all-ones code word -> {symbol: code length}"""
    bits, vals, _ = gen_optimal_table(counts)
    got_bits = list(h.bits)
    n = sum(got_bits)
    assert h.present == 1
    assert got_bits == bits and list(h.vals[:n]) == vals and not any(h.vals[n:])
    assert sum(b * 2 ** (16 - L) for L, b in zip(range(1, 17), got_bits)) < 2 ** 16   # Kraft, the all-ones word left out
    lens = code_lengths(got_bits, vals)
    assert all(counts[s] > 0 for s in lens) and all(s in lens for s in range(len(counts)) if counts[s] > 0)
    return lens


def check_tables(ht, coefs):
    """all four tables of one image; returns the un-stuffed bit count they give"""
    hist, total = symbol_hist(coefs)
    for cls in (0, 1):
        dcl = check_table(ht[0][cls], hist[cls, :16])
        acl = check_table(ht[1][cls], hist[cls, 16:])
        total += sum(int(hist[cls, s]) * L for s, L in dcl.items()) + sum(int(hist[cls, 16 + s]) * L for s, L in acl.items())
    return total


def with_tables(header, ht):
    """the header with its four DHT segments replaced by the tables (same order, lengths from the tables)"""
    out, i = bytearray(header[:2]), 2
    while i < len(header):
        m, ln = header[i + 1], (header[i + 2] << 8) | header[i + 3]
        seg = header[i:i + 2 + ln]
        out += dht(seg[4], ht[seg[4] >> 4][seg[4] & 15]) if m == 0xC4 else seg
        i += 2 + ln
    return bytes(out)


def opt_file(oracle, W, H, gray, scan, ht):
    return with_tables(oracle.header(W, H, gray=gray), ht) + scan + b"\xff\xd9"


def dev_opt_entropy(ctx, coefs, W, H, nimg=1):
    dc = to_dev(np.ascontiguousarray(coefs, dtype=np.int16))
    slot = max(W * H * 3, 10240)
    out = torch.zeros((nimg, slot), dtype=torch.uint8, device="cuda")
    nbytes = torch.zeros(nimg, dtype=torch.int64, device="cuda")
    nbits = torch.zeros(nimg, dtype=torch.int64, device="cuda")
    d_ht = torch.zeros(nimg * HB, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.entropy_encode_optimized_dev(dc, W, H, nimg, False, out, slot, d_ht, nbytes, nbits, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    nb, o, h = nbytes.cpu().numpy(), out.cpu().numpy(), d_ht.cpu().numpy()
    return ([o[i, : nb[i]].tobytes() if nb[i] >= 0 else None for i in range(nimg)], nbits.cpu().numpy(),
            [J.huff_tables(h[i * HB:(i + 1) * HB]) for i in range(nimg)])


# ---- 1 + 4: tables, bit count, never longer than Annex K ---------------------------------------------
@pytest.mark.parametrize("W,H", TABLE_SIZES)
@pytest.mark.parametrize("family", [0, 1, 2])
@pytest.mark.parametrize("gray", [False, True])
def test_tables_match_reference(ctx, oracle, W, H, family, gray):
    r, g, b = planes(family, W, H)
    coefs = oracle.coefs(r, g, b, W, H, gray=gray)
    scan, nbits, ht = ctx.encode_optimized(r, g, b, W, H, gray=gray)
    assert nbits == check_tables(ht, coefs)
    _, nbits_k = ctx.encode(r, g, b, W, H, gray=gray)
    assert nbits <= nbits_k
    if gray:   # chroma AC holds EOB alone: one real symbol, the 1-bit code 0
        assert list(ht[1][1].bits) == [1] + [0] * 15 and ht[1][1].vals[0] == 0


# ---- 2: length limiting and coefficients without a baseline code ---------------------------------------
def test_length_limiting(ctx, oracle):
    coefs, W, H = fibonacci_coefs()
    hist, _ = symbol_hist(coefs)
    assert max(gen_optimal_table(hist[0, 16:])[2]) > 16   # the unconstrained code is longer than 16 bits
    scans, nbits, hts = dev_opt_entropy(ctx, coefs, W, H)
    ht = hts[0]
    assert nbits[0] == check_tables(ht, coefs)
    assert max(L for L in range(1, 17) if ht[1][0].bits[L - 1]) == 16
    assert (oracle.decode_coefs(opt_file(oracle, W, H, False, scans[0], ht)) == coefs).all()


def test_coefficient_without_code_reports_overflow(ctx):
    W, H = 32, 16
    coefs = np.zeros((2, 6, 64), np.int16)
    coefs[1, 2, 5] = 1024   # an 11-bit AC value
    scans, nbits, _ = dev_opt_entropy(ctx, coefs, W, H)
    assert scans[0] is None and nbits[0] == -1


# ---- 3: the segment is the right encoding ---------------------------------------------------------------
@pytest.mark.parametrize("W,H", [(17, 33), (200, 120), (1920, 1080)])
@pytest.mark.parametrize("family", [0, 1, 2])
@pytest.mark.parametrize("gray", [False, True])
def test_file_decodes_like_annex_k_file(ctx, oracle, W, H, family, gray):
    from PIL import Image
    r, g, b = planes(family, W, H)
    scan, _, ht = ctx.encode_optimized(r, g, b, W, H, gray=gray)
    f = opt_file(oracle, W, H, gray, scan, ht)
    assert (oracle.decode_coefs(f) == oracle.coefs(r, g, b, W, H, gray=gray)).all()
    ref = oracle.encode(r, g, b, W, H, gray=gray)
    assert len(f) <= len(ref)
    a, k = np.asarray(Image.open(io.BytesIO(f))), np.asarray(Image.open(io.BytesIO(ref)))
    assert a.shape == k.shape and (a == k).all()


@pytest.mark.parametrize("W,H", [(200, 120), (1920, 1080), (3840, 2160)])
@pytest.mark.parametrize("family", [0, 1])
@pytest.mark.parametrize("gray", [False, True])
def test_device_round_trip_matches_annex_k(ctx, W, H, family, gray):
    r, g, b = planes(family, W, H)
    scan, _, ht = ctx.encode_optimized(r, g, b, W, H, gray=gray)
    scan_k, _ = ctx.encode(r, g, b, W, H, gray=gray)
    got = ctx.decode(scan, J.optimized_frame(W, H, ht), gray=gray)
    want = ctx.decode(scan_k, J.default_frame(W, H), gray=gray)
    assert all((x == y).all() for x, y in zip(got, want))
    if W == 3840:
        print("4K family %d gray %d: %d bytes Annex K, %d optimised (%.2f %% smaller)" %
              (family, gray, len(scan_k), len(scan), 100.0 * (1 - len(scan) / len(scan_k))))


# ---- 5: batch, determinism, both transform kernels, guard zones ------------------------------------------
def test_batch_equals_single_calls(ctx):
    W, H, n, G = 200, 120, 11, 4096
    imgs = [planes(i % 3, W, H, frame=i) for i in range(n)]
    d_in = to_dev(np.stack([np.stack(p) for p in imgs], 1))   # [3][n][H][W]
    slot = W * H * 3
    sp = torch.cuda.current_stream().cuda_stream

    def run_batch():
        scan = torch.full((2 * G + n * slot,), 0xA5, dtype=torch.uint8, device="cuda")
        ht = torch.full((2 * G + n * HB,), 0x5A, dtype=torch.uint8, device="cuda")
        nbytes = torch.zeros(n, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        ctx.encode_batch_optimized_dev(d_in[0], d_in[1], d_in[2], W, H, n, False, scan[G:].data_ptr(), slot, ht[G:].data_ptr(),
                                       nbytes, stream=sp)
        torch.cuda.synchronize()
        s, h, nb = scan.cpu().numpy(), ht.cpu().numpy(), nbytes.cpu().numpy()
        assert (s[:G] == 0xA5).all() and (s[G + n * slot:] == 0xA5).all()
        assert (h[:G] == 0x5A).all() and (h[G + n * HB:] == 0x5A).all()
        return [s[G + i * slot: G + i * slot + nb[i]].tobytes() for i in range(n)], h[G:G + n * HB].tobytes()

    first = run_batch()
    assert run_batch() == first
    try:
        ctx.set_option(capi.OPT_TRANSFORM, 1)
        assert run_batch() == first
    finally:
        ctx.set_option(capi.OPT_TRANSFORM, 0)
    for i, (r, g, b) in enumerate(imgs):
        scan, _, ht = ctx.encode_optimized(r, g, b, W, H)
        assert scan == first[0][i] and bytes(ht) == first[1][i * HB:(i + 1) * HB]


def test_entropy_stage_without_side_information(ctx, oracle):
    # the per-stage entry point reads every coefficient group (no forward-transform side information)
    W, H = 200, 120
    r, g, b = planes(0, W, H)
    coefs = oracle.coefs(r, g, b, W, H)
    scans, nbits, hts = dev_opt_entropy(ctx, coefs, W, H)
    scan, nb, ht = ctx.encode_optimized(r, g, b, W, H)
    assert scans[0] == scan and nbits[0] == nb and bytes(hts[0]) == bytes(ht)


# ---- 6: CLI ------------------------------------------------------------------------------------------
def write_ppm(path, r, g, b):
    H, W = r.shape
    rgb = np.stack([r, g, b], -1).reshape(-1, 3)
    path.write_text("P3\n%d %d\n255\n" % (W, H) + "\n".join("%d %d %d" % tuple(p) for p in rgb) + "\n")


@pytest.mark.parametrize("gray", [False, True])
def test_cli_optimize(tmp_path, oracle, gray):
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "jpezy_b200", "cli"), "-s"])
    enc, dec = os.path.join(BIN, "jpezy_encode"), os.path.join(BIN, "jpezy_decode")
    W, H = 129, 65
    r, g, b = planes(0, W, H)
    src = tmp_path / "in.ppm"
    write_ppm(src, r, g, b)
    flags = ["--gray"] if gray else []
    for name, extra in (("k", []), ("o", ["--optimize"])):
        p = subprocess.run([enc, str(src), str(tmp_path / (name + ".jpg")), *extra, *flags], capture_output=True, text=True)
        assert p.returncode == 0, p.stderr
        q = subprocess.run([dec, str(tmp_path / (name + ".jpg")), str(tmp_path / (name + ".ppm")), *flags], capture_output=True, text=True)
        assert q.returncode == 0, q.stderr
    fk, fo = (tmp_path / "k.jpg").read_bytes(), (tmp_path / "o.jpg").read_bytes()
    assert fk == oracle.encode(r, g, b, W, H, gray=gray)
    assert (oracle.decode_coefs(fo) == oracle.coefs(r, g, b, W, H, gray=gray)).all()
    assert (tmp_path / "o.ppm").read_text() == (tmp_path / "k.ppm").read_text()
    assert len(fo) < len(fk)
