"""CPU tests that pin Oracle.pixels_from_coefs -- the reference decoder's pixel stage (dequant, idct, replication, make_rgb) on
given coefficients, the yardstick of tests/test_inverse_reference_gpu.py -- to the oracle's file decoder, which
tests/test_oracle_vs_ref.py pins to the reference's own code: both run the same per-MCU code, so decoding a file's
coefficients must give the file's pixels, in colour and gray output, for every sampling layout the device decoder takes."""
import hashlib
import io
import json
import os

import numpy as np
import pytest

import jpezy_b200 as J

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
VEC = json.load(open(os.path.join(G, "oracle_vectors.json")))

# sampling factors (hs, vs) per layout
LAYOUTS = {"444": ((1, 1, 1), (1, 1, 1)), "422": ((2, 1, 1), (1, 1, 1)), "440": ((1, 1, 1), (2, 1, 1)), "gray1": ((1,), (1,)),
           "420": ((2, 1, 1), (2, 1, 1))}


def dqt_tables(f):
    """natural-order quantisation tables of the file by Tq, and the Tq of every component (SOF0)"""
    zz = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28, 35, 42,
          49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]
    tabs, tq, p = {}, [], 2
    while p < len(f):
        assert f[p] == 0xFF
        m, ln = f[p + 1], int.from_bytes(f[p + 2: p + 4], "big")
        seg = f[p + 4: p + 2 + ln]
        if m == 0xDB:
            i = 0
            while i < len(seg):
                pq, t = seg[i] >> 4, seg[i] & 15
                n = 2 if pq else 1
                vals = [int.from_bytes(seg[i + 1 + k * n: i + 1 + (k + 1) * n], "big") for k in range(64)]
                nat = [0] * 64
                for k in range(64):
                    nat[zz[k]] = vals[k]
                tabs[t] = nat
                i += 1 + 64 * n
        elif m == 0xC0:
            tq = [seg[6 + 3 * c + 2] for c in range(seg[5])]
        elif m == 0xDA:
            break
        p += 2 + ln
    return np.array([tabs[t] for t in tq], dtype=np.uint16)


def pillow_file(layout, W, H):
    PIL = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(W * 7 + H)
    y, x = np.mgrid[0:H, 0:W]
    img = np.stack([(x * 3 + y) % 256, (x + 2 * y) % 256, (x * y // 7) % 256], -1) // 2 + rng.integers(0, 128, (H, W, 3))
    img = img.clip(0, 255).astype(np.uint8)
    buf = io.BytesIO()
    if layout == "gray1":
        PIL.fromarray(img[..., 0], "L").save(buf, "JPEG", quality=85)
    else:
        sub = {"444": 0, "440": 1, "422": 1, "420": 2}[layout]
        PIL.fromarray(img, "RGB").save(buf, "JPEG", quality=70, subsampling=sub)
    f = bytearray(buf.getvalue())
    if layout == "440":
        # Pillow writes no 4:4:0: a 4:2:2 scan (Y Y Cb Cr per MCU) read with luma sampling 1x2 is one, of the same MCU count when
        # W and H are multiples of 16
        p = f.index(b"\xff\xc0")
        assert f[p + 11] == 0x21
        f[p + 11] = 0x12
    return bytes(f)


@pytest.mark.parametrize("name", sorted(VEC))
@pytest.mark.parametrize("gray_out", [False, True])
def test_pixels_from_coefs_equals_file_decoder_on_golden_vectors(oracle, name, gray_out):
    v = VEC[name]
    r, g, b = J.synth.image(v["family"], v["W"], v["H"])
    f = oracle.encode(r, g, b, v["W"], v["H"], gray=v["gray"])
    assert hashlib.sha256(f).hexdigest() == v["file_sha256"]
    _, qy, qc, _, _ = oracle.tables()
    want = oracle.decode(f, gray=gray_out)[2:]
    got = oracle.pixels_from_coefs(oracle.decode_coefs(f), v["W"], v["H"], np.stack([qy, qc, qc]), gray=gray_out)
    for a, w in zip(got, want):
        assert a.shape == w.shape and (a == w).all()


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
@pytest.mark.parametrize("W,H", [(70, 45), (8, 8), (129, 257), (48, 32)])
@pytest.mark.parametrize("gray_out", [False, True])
def test_pixels_from_coefs_equals_file_decoder_on_pillow_files(oracle, layout, W, H, gray_out):
    if layout == "440" and (W % 16 or H % 16):
        pytest.skip("4:4:0 files are patched 4:2:2 files: same MCU count only when W and H are multiples of 16")
    f = pillow_file(layout, W, H)
    hs, vs = LAYOUTS[layout]
    _, _, _, nc, fhs, fvs, nblk = oracle.layout(f)
    assert (fhs, fvs) == (hs, vs)
    c = oracle.decode_coefs(f)
    assert c.size == nblk * 64
    want = oracle.decode(f, gray=gray_out)[2:]
    got = oracle.pixels_from_coefs(c, W, H, dqt_tables(f), ncomp=nc, hs=hs, vs=vs, gray=gray_out)
    for a, w in zip(got, want):
        assert a.shape == w.shape and (a == w).all()


def test_pixels_from_coefs_keeps_dc_values_beyond_int16(oracle):
    """int32 coefficients: a DC of 40000 (reachable by a stream whose DC differences keep one sign) gives a luma sample of
    40000 * 16 / 8 + 128, saturated to 255 in gray output; the same block with DC wrapped to int16 gives 0"""
    W = H = 16
    c = np.zeros((1, 6, 64), np.int32)
    c[0, 0, 0] = 40000
    q = np.ones((3, 64), np.uint16) * 16
    r, _, _ = oracle.pixels_from_coefs(c, W, H, q, gray=True)
    assert (r.reshape(16, 16)[:8, :8] == 255).all()
    c[0, 0, 0] = np.int16(np.int32(40000).astype(np.int16))
    r, _, _ = oracle.pixels_from_coefs(c, W, H, q, gray=True)
    assert (r.reshape(16, 16)[:8, :8] == 0).all()
    f = oracle.header(W, H) + oracle.scan_from_coefs(np.clip(c, -2047, 2047)) + b"\xff\xd9"
    assert (oracle.decode_coefs(f) == np.clip(c, -2047, 2047)).all()
