"""-m gpu: every inverse-transform route of the device decoder against the reference decoder's pixel stage
(Oracle.pixels_from_coefs, pinned to the file decoder by tests/test_oracle_pixels.py) on coefficients no encoder writes:
DC-only warps, pruned and barely unpruned flowgraphs, dense full-range blocks whose samples leave the int16 range, negative
samples, exact ties that only the reference's FP64 rounding decides, wild chroma -- under Annex K, flat, distinct-chroma and 16-bit
quantisation tables, at ragged and full-HD geometry.  Bar: zero differing samples.  The entropy side gets the same coefficients
through files: entropy_decode_dev must return them unchanged, and a DC that walks past the int16 range is reported per image."""
import numpy as np
import pytest
import torch

import jpezy_b200 as J
from jpezy_b200 import capi
from gpu_util import Guarded

pytestmark = pytest.mark.gpu

LAYOUTS = {"420": ((2, 1, 1), (2, 1, 1)), "444": ((1, 1, 1), (1, 1, 1)), "422": ((2, 1, 1), (1, 1, 1)), "440": ((1, 1, 1), (2, 1, 1)),
           "gray1": ((1,), (1,))}
FAMILIES = ["dc_only", "low", "mostly_pruned", "sparse", "dense", "neg_dc", "ties", "chroma_wild"]
TABLES = ["annexk", "ones", "all255", "distinct", "bits16"]
EAGAIN, EUNSUPPORTED = 9, 8


def qtables(oracle, kind):
    """three natural-order tables (Y, Cb, Cr)"""
    _, qy, qc, _, _ = oracle.tables()
    if kind == "annexk":
        return np.stack([qy, qc, qc]).astype(np.uint16)
    if kind == "ones":
        return np.ones((3, 64), np.uint16)
    if kind == "all255":
        return np.full((3, 64), 255, np.uint16)
    if kind == "distinct":
        i = np.arange(64)
        return np.stack([qy, 11 + 3 * (i % 8) + (i // 8), 29 + (i % 8) + 5 * (i // 8)]).astype(np.uint16)
    rng = np.random.default_rng(16)           # 16-bit DQT values (Pq = 1)
    return rng.integers(1, 65536, size=(3, 64)).astype(np.uint16)


def geometry(W, H, layout):
    hs, vs = LAYOUTS[layout]
    hu, vu = -(-W // (8 * max(hs))), -(-H // (8 * max(vs)))
    return hs, vs, hu * vu, sum(a * b for a, b in zip(hs, vs))


def coefficients(family, nmcu, nb, ny, q, seed):
    """[nmcu, nb, 64] int32 zig-zag coefficients in scan order (|AC| <= 1023 and |DC| <= 1023, so that Annex K Huffman tables can
    code them); q: the three tables"""
    rng = np.random.default_rng(seed)
    c = np.zeros((nmcu, nb, 64), np.int32)
    n = nmcu * nb
    flat = c.reshape(n, 64)
    if family == "dc_only":                  # whole warps of DC-only blocks, values across the whole DC range
        flat[:, 0] = rng.integers(-1023, 1024, n)
    elif family == "low":                    # nothing beyond zig-zag position 7: the pruned flowgraphs
        flat[:, 0] = rng.integers(-300, 300, n)
        flat[:, 1:8] = rng.integers(-60, 61, (n, 7))
    elif family == "mostly_pruned":          # as "low", and one block in eight reaches a random position in 8..63
        flat[:, 0] = rng.integers(-300, 300, n)
        flat[:, 1:8] = rng.integers(-40, 41, (n, 7))
        hit = np.arange(n)[rng.integers(0, 8) :: 8]
        flat[hit, rng.integers(8, 64, hit.size)] = rng.integers(-200, 201, hit.size)
    elif family == "sparse":
        flat[:] = rng.integers(-30, 31, (n, 64)) * (rng.random((n, 64)) < 0.15)
        flat[:, 0] = rng.integers(-200, 200, n)
    elif family == "dense":                  # full range: samples far beyond int16, the fix-up queue of a tile overflows
        flat[:] = rng.integers(-1023, 1024, (n, 64))
    elif family == "neg_dc":                 # negative samples, where the reference's truncation is not floor
        flat[:, 0] = rng.integers(-1023, -400, n)
        flat[:, 1:20] = rng.integers(-25, 26, (n, 19)) * (rng.random((n, 19)) < 0.5)
    elif family == "ties":
        # DC + one coefficient at (u, v) = (4, 0) or (0, 4): every sample is (DC q0 +- c q) / 8 + 128 in exact arithmetic, an integer
        # when both signs are 0 mod 8; the reference's FP64 rounding then decides
        comp = np.array([0 if k < ny else k - ny + 1 for k in range(nb)] * nmcu)
        zz_u4, zz_v4 = 14, 10                # zig-zag positions of natural 4 (v 0, u 4) and 32 (v 4, u 0)
        for i in range(n):
            qq = q[comp[i]]
            pos, nat = (zz_u4, 4) if rng.random() < 0.5 else (zz_v4, 32)
            for _ in range(10000):
                dc, ac = int(rng.integers(-1023, 1024)), int(rng.integers(-1023, 1024))
                if ac and (dc * int(qq[0]) + ac * int(qq[nat])) % 8 == 0 and (dc * int(qq[0]) - ac * int(qq[nat])) % 8 == 0:
                    flat[i, 0], flat[i, pos] = dc, ac
                    break
    elif family == "chroma_wild":            # mid luma, chroma far outside [0, 255] or on the near-integer G boundary
        flat[:, 0] = rng.integers(-20, 20, n)
        ch = c[:, ny:, :].reshape(-1, 64)
        ch[:, 0] = rng.integers(-1023, 1024, ch.shape[0])
        ch[:, 1:4] = rng.integers(-3, 4, (ch.shape[0], 3))
        c[:, ny:, :] = ch.reshape(nmcu, nb - ny, 64)
    assert np.abs(c).max() <= 1023
    return c


def frame_for(W, H, layout, q, restart_interval=0):
    hs, vs = LAYOUTS[layout]
    f = J.default_frame(W, H)
    f.ncomp = len(hs)
    for i in range(len(hs)):
        f.hs[i], f.vs[i], f.tq[i] = hs[i], vs[i], i
        for k in range(64):
            f.qt[i][k] = int(q[i][k])
    f.restart_interval = restart_interval
    return f


def reference(oracle, c, W, H, layout, q, gray):
    hs, vs = LAYOUTS[layout]
    return oracle.pixels_from_coefs(c, W, H, q[: len(hs)], ncomp=len(hs), hs=hs, vs=vs, gray=gray)


def check_planes(got, want, what):
    for k, (a, w) in enumerate(zip(got, want)):
        a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
        nd = int((a != w).sum())
        assert nd == 0, "%s: %d of %d samples of plane %d differ from the reference decoder" % (what, nd, w.size, k)


def run_inverse(ctx, cs, frame, gray, route, coef_offset=0, plane_offset=0):
    """transform_inv_dev on nimg images of coefficients; -> per image the three planes"""
    nimg = len(cs)
    pl = capi.plane_bytes(frame)
    d = Guarded(sum(x.size for x in cs), torch.int16, offset=coef_offset)
    d.view.copy_(torch.from_numpy(np.concatenate([x.reshape(-1) for x in cs]).astype(np.int16)).cuda())
    out = [Guarded(nimg * pl, torch.uint8, fill=0x5A, offset=plane_offset) for _ in range(3)]
    ctx.set_option(capi.OPT_TRANSFORM, 1 if route == "f64" else 0)
    try:
        ctx.transform_inv_dev(d.view, frame, nimg, gray, out[0].view, out[1].view, out[2].view, pl,
                              stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    finally:
        ctx.set_option(capi.OPT_TRANSFORM, 0)
    assert d.intact() and all(o.intact() for o in out), "a guard zone was written"
    return [[o.view[i * pl: (i + 1) * pl] for o in out] for i in range(nimg)]


# route -> (layouts, coefficient byte offset, plane byte offset); the selection of launch_inv (capi_decode.inc)
ROUTES = {"inv2": (["420"], 0, 0),                        # k_inv_transform2<8>: 4:2:0, every buffer 16-byte aligned
          "inv1": (["420"], 0, 1),                        # k_inv_transform: 4:2:0, planes 1 byte off
          "general": (["444", "422", "440", "gray1"], 0, 0),   # k_idct_blocks + k_colour_general
          "f64": (list(LAYOUTS), 0, 0),                    # k_inv_transform_f64: JPEZYB200_OPT_TRANSFORM = 1
          "f64_unaligned": (["444", "422", "440", "gray1"], 2, 0)}   # general layouts whose coefficients are not 16-byte aligned
GEOMS = [(200, 120), (1, 1), (256, 48)]     # W % 16 != 0 (13 MCUs a row: not a whole number of 8-MCU tiles, H % 16 != 0); 1x1; W % 16 == 0


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("route", sorted(ROUTES))
def test_inverse_route_matches_reference(ctx, oracle, route, family):
    """three images of different content per call; layouts, tables and geometry rotate with the family so that every route
    meets every table kind and both output modes"""
    layouts, coff, poff = ROUTES[route]
    fi = FAMILIES.index(family)
    for li, layout in enumerate(layouts):
        tkind = TABLES[(fi + li) % len(TABLES)]
        q = qtables(oracle, tkind)
        W, H = GEOMS[(fi + li) % len(GEOMS)]
        gray = (fi + li) % 2 == 1
        hs, vs, nmcu, nb = geometry(W, H, layout)
        cs = [coefficients(family, nmcu, nb, hs[0] * vs[0], q, seed=1000 * fi + 10 * li + i) for i in range(3)]
        frame = frame_for(W, H, layout, q)
        before = ctx.stat(capi.STAT_GUARD_INV)
        got = run_inverse(ctx, cs, frame, gray, route, coff, poff)
        for i in range(3):
            check_planes(got[i], reference(oracle, cs[i], W, H, layout, q, gray),
                         "%s %s %s %dx%d tables %s gray %d image %d" % (route, layout, family, W, H, tkind, gray, i))
        if family == "ties":
            assert ctx.stat(capi.STAT_GUARD_INV) > before, "no sample took the exact-order tier"


@pytest.mark.parametrize("tkind", TABLES)
@pytest.mark.parametrize("route", sorted(ROUTES))
@pytest.mark.parametrize("gray", [False, True])
def test_inverse_route_every_table_kind(ctx, oracle, route, tkind, gray):
    """dense and sparse blocks side by side (per-block routing inside a tile) under every table kind"""
    layouts, coff, poff = ROUTES[route]
    q = qtables(oracle, tkind)
    W, H = 72, 40
    for li, layout in enumerate(layouts):
        hs, vs, nmcu, nb = geometry(W, H, layout)
        ny = hs[0] * vs[0]
        a = coefficients("sparse", nmcu, nb, ny, q, seed=7 + li)
        b = coefficients("dense", nmcu, nb, ny, q, seed=8 + li)
        if tkind == "bits16":       # keep the reference's int products c * q far below 2^31
            b = b // 64
        mix = np.where((np.arange(nmcu * nb) % 5 == 0).reshape(nmcu, nb, 1), b, a)
        got = run_inverse(ctx, [mix], frame_for(W, H, layout, q), gray, route, coff, poff)
        check_planes(got[0], reference(oracle, mix, W, H, layout, q, gray), "%s %s tables %s gray %d" % (route, layout, tkind, gray))


@pytest.mark.parametrize("route", ["inv2", "inv1", "f64"])
@pytest.mark.parametrize("family", ["dense", "sparse"])
def test_inverse_full_hd_frame(ctx, oracle, route, family):
    W, H = 1920, 1088
    q = qtables(oracle, "annexk")
    hs, vs, nmcu, nb = geometry(W, H, "420")
    c = coefficients(family, nmcu, nb, 4, q, seed=3)
    got = run_inverse(ctx, [c], frame_for(W, H, "420", q), False, route, 0, ROUTES[route][2])
    check_planes(got[0], reference(oracle, c, W, H, "420", q, False), "%s %s 1920x1088" % (route, family))


def scans(oracle, cs, restart_interval=0):
    return [oracle.scan_from_coefs(c, restart_interval=restart_interval) for c in cs]


def upload_scans(ss):
    slot = max(len(s) for s in ss) + 64
    buf = np.zeros((len(ss), slot), np.uint8)
    for i, s in enumerate(ss):
        buf[i, : len(s)] = np.frombuffer(s, np.uint8)
    return torch.from_numpy(buf).cuda(), slot, np.array([len(s) for s in ss], np.uint64)


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("gray", [False, True])
def test_fused_decode_matches_reference(ctx, oracle, family, gray):
    """files made from the coefficients (Annex K Huffman tables): the fused decode with the dense DC array, through
    jpezyb200_decode and decode_batch_dev2 (three images, different content); entropy_decode_dev returns the very coefficients
    (full-range blocks: 10-bit AC codes, ZRL chains, blocks without EOB) or EAGAIN, never something else"""
    fi = FAMILIES.index(family)
    tkind = ["annexk", "ones", "all255", "distinct", "bits16"][fi % 5]
    q = qtables(oracle, tkind)
    W, H = [(200, 120), (256, 48), (8, 8)][fi % 3]
    _, _, nmcu, nb = geometry(W, H, "420")
    cs = [coefficients(family, nmcu, nb, 4, q, seed=500 + 10 * fi + i) for i in range(3)]
    if tkind == "bits16":
        cs = [c // 64 for c in cs]
    frame = frame_for(W, H, "420", q)
    want = [reference(oracle, c, W, H, "420", q, gray) for c in cs]
    ss = scans(oracle, cs)
    for i in range(3):
        check_planes(ctx.decode(ss[i], frame, gray=gray), want[i], "jpezyb200_decode %s image %d" % (family, i))
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
            check_planes([o.view[i * pl: (i + 1) * pl] for o in out], want[i], "decode_batch_dev2 %s image %d" % (family, i))
    assert all(o.intact() for o in out)
    coefs = Guarded(3 * nmcu * nb * 64, torch.int16, fill=0x7777)
    st.fill_(-1)
    ctx.entropy_decode_dev(d_scan, slot, nbytes, 3, frame, coefs.view, st, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    got = coefs.view.cpu().numpy().reshape(3, nmcu, nb, 64)
    for i, s in enumerate(st.cpu().tolist()):
        assert s in (0, EAGAIN)
        if s == 0:
            nd = int((got[i] != cs[i]).sum())
            assert nd == 0, "entropy_decode_dev: %d coefficients of image %d differ from those the file was made from" % (nd, i)
    assert coefs.intact()


def dc_walk(nmcu, seed, restart_interval):
    """4:2:0 coefficients whose luma DC keeps climbing by 2000 a block (from 0 again in every restart interval): past +32767 after
    17 blocks"""
    rng = np.random.default_rng(seed)
    c = np.zeros((nmcu, 6, 64), np.int32)
    per = 4 * (restart_interval or nmcu)
    c[:, :4, 0] = ((np.arange(nmcu * 4) % per) * 2000).reshape(nmcu, 4)
    c[:, :, 1:6] = rng.integers(-5, 6, (nmcu, 6, 5))
    return c


@pytest.mark.parametrize("restart_interval", [0, 8])
def test_dc_beyond_int16_is_reported_on_that_image_only(ctx, oracle, restart_interval):
    """the reference keeps the DC predictor in an int and decodes such a stream; the int16 coefficient format cannot carry it, so
    the device reports JPEZYB200_EUNSUPPORTED for that image and decodes the others of the batch correctly"""
    W, H = 128, 32                              # 16 MCUs, 64 luma blocks: the DC reaches 126000
    q = qtables(oracle, "annexk")
    _, _, nmcu, nb = geometry(W, H, "420")
    cs = [coefficients("sparse", nmcu, nb, 4, q, seed=90), dc_walk(nmcu, 91, restart_interval), coefficients("low", nmcu, nb, 4, q, seed=92)]
    assert cs[1].max() > 32767
    frame = frame_for(W, H, "420", q, restart_interval)
    ss = scans(oracle, cs, restart_interval)
    d_scan, slot, nbytes = upload_scans(ss)
    pl = capi.plane_bytes(frame)
    sp = torch.cuda.current_stream().cuda_stream
    # fused decode (dense DC array, or the restart-interval decoder)
    out = [torch.zeros(3 * pl, dtype=torch.uint8, device="cuda") for _ in range(3)]
    st = torch.full((3,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    ctx.decode_batch_dev(d_scan, slot, nbytes, 3, frame, False, out[0], out[1], out[2], pl, st, stream=sp)
    torch.cuda.synchronize()
    assert st.cpu().tolist() == [0, EUNSUPPORTED, 0]
    for i in (0, 2):
        check_planes([o[i * pl: (i + 1) * pl] for o in out], reference(oracle, cs[i], W, H, "420", q, False), "fused image %d" % i)
    # per-stage decode
    coefs = torch.zeros(3 * nmcu * nb * 64, dtype=torch.int16, device="cuda")
    st.fill_(-1)
    ctx.entropy_decode_dev(d_scan, slot, nbytes, 3, frame, coefs, st, stream=sp)
    torch.cuda.synchronize()
    assert st.cpu().tolist() == [0, EUNSUPPORTED, 0]
    got = coefs.cpu().numpy().reshape(3, nmcu, nb, 64)
    assert (got[0] == cs[0]).all() and (got[2] == cs[2]).all()
    # the host entry point returns the status instead of wrapped pixels
    with pytest.raises(J.JpezyError) as e:
        ctx.decode(ss[1], frame)
    assert e.value.code == EUNSUPPORTED
    check_planes(ctx.decode(ss[0], frame), reference(oracle, cs[0], W, H, "420", q, False), "jpezyb200_decode")
