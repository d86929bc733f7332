"""-m gpu: what every encode and decode entry point of the C ABI launches, and what it returns for bad arguments.

Each entry point runs twice on a fresh context with seeded inputs, at the C1 size (512x512) and at 1920x1080.  The kernels
each call launches (JPEZYB200_STAT_KERNEL_LAUNCHES) are pinned for both calls: the first builds the context's per-frame
tables, the second finds them cached.  A table of bad arguments pins the status code of each entry point.  Both hold the
host code of the C ABI to the launches and the argument checks it had before it was restructured."""
import ctypes as C

import numpy as np
import pytest
import torch

import jpezy_b200 as J
from jpezy_b200 import capi
from jpezy_b200.capi import ECAPACITY, ECORRUPT, EINVAL, OK, _dp

pytestmark = pytest.mark.gpu

SIZES = [(512, 512), (1920, 1080)]
NIMG = 2          # images of the batch forms
HB = capi.HUFF_TABLES_BYTES


class Inputs:
    """NIMG seeded frames of one size, on the host and on the device, with their Annex K segments and coefficients"""

    def __init__(self, W, H):
        self.W, self.H = W, H
        frames = [J.synth.image(0, W, H, frame=1 + i) for i in range(NIMG)]
        self.host = [np.ascontiguousarray(np.stack([f[c].reshape(-1) for f in frames])) for c in range(3)]   # [NIMG, W*H] each
        self.dev = [torch.from_numpy(a).cuda() for a in self.host]
        self.frame = J.default_frame(W, H)
        self.need = capi.plane_bytes(self.frame)
        self.slot = max(3 * W * H, 10240)
        self.nmcu = capi.num_mcus(W, H)
        self.VU = (H + 15) // 16
        c = J.Context(0)
        try:
            self.coefs = torch.zeros((NIMG, self.nmcu * 384), dtype=torch.int16, device="cuda")
            self.d_scan = torch.zeros((NIMG, self.slot), dtype=torch.uint8, device="cuda")
            self.d_bytes = torch.zeros(NIMG, dtype=torch.int64, device="cuda")
            torch.cuda.synchronize()
            c.transform_fwd_dev(*self.dev, W, H, NIMG, False, self.coefs)
            c.entropy_encode_dev(self.coefs, W, H, NIMG, False, self.d_scan, self.slot, self.d_bytes)
            torch.cuda.synchronize()
        finally:
            c.close()
        self.h_bytes = self.d_bytes.cpu().numpy().astype(np.uint64)
        self.h_scan = self.d_scan.cpu().numpy()
        self.scan0 = self.h_scan[0, : int(self.h_bytes[0])].tobytes()

    def planes_out(self, nimg=NIMG):
        return [torch.empty(nimg * self.need, dtype=torch.uint8, device="cuda") for _ in range(3)]


_INPUTS = {}


def inputs(W, H):
    if (W, H) not in _INPUTS:
        _INPUTS[(W, H)] = Inputs(W, H)
    return _INPUTS[(W, H)]


# ---- one valid call of each entry point -------------------------------------------------------------------------------
def run_encode(c, x):
    c.encode(x.host[0][0], x.host[1][0], x.host[2][0], x.W, x.H)


def run_encode_optimized(c, x):
    c.encode_optimized(x.host[0][0], x.host[1][0], x.host[2][0], x.W, x.H)


def run_encode_batch(c, x):
    out = np.empty(NIMG * x.slot, np.uint8)
    nb = np.zeros(NIMG, np.uint64)
    c.encode_batch(*x.host, x.W, x.H, NIMG, False, out, x.slot, nb)


def run_encode_batch_dev(c, x):
    out = torch.empty((NIMG, x.slot), dtype=torch.uint8, device="cuda")
    nb = torch.empty(NIMG, dtype=torch.int64, device="cuda")
    c.encode_batch_dev(*x.dev, x.W, x.H, NIMG, False, out, x.slot, nb)


def run_encode_batch_optimized_dev(c, x):
    out = torch.empty((NIMG, x.slot), dtype=torch.uint8, device="cuda")
    nb = torch.empty(NIMG, dtype=torch.int64, device="cuda")
    ht = torch.empty(NIMG * HB, dtype=torch.uint8, device="cuda")
    c.encode_batch_optimized_dev(*x.dev, x.W, x.H, NIMG, False, out, x.slot, ht, nb)


def run_transform_fwd_dev(c, x):
    coefs = torch.empty_like(x.coefs)
    c.transform_fwd_dev(*x.dev, x.W, x.H, NIMG, False, coefs)


def run_entropy_encode_dev(c, x):
    out = torch.empty((NIMG, x.slot), dtype=torch.uint8, device="cuda")
    nb = torch.empty(NIMG, dtype=torch.int64, device="cuda")
    c.entropy_encode_dev(x.coefs, x.W, x.H, NIMG, False, out, x.slot, nb)


def run_entropy_encode_optimized_dev(c, x):
    out = torch.empty((NIMG, x.slot), dtype=torch.uint8, device="cuda")
    nb = torch.empty(NIMG, dtype=torch.int64, device="cuda")
    ht = torch.empty(NIMG * HB, dtype=torch.uint8, device="cuda")
    c.entropy_encode_optimized_dev(x.coefs, x.W, x.H, NIMG, False, out, x.slot, ht, nb)


def shard_buffers():
    s = dict(last_dc=torch.zeros(3, dtype=torch.int32, device="cuda"), dc_init=torch.zeros(3, dtype=torch.int32, device="cuda"),
             info=torch.zeros(2, dtype=torch.int64, device="cuda"), nbytes=torch.zeros(1, dtype=torch.int64, device="cuda"),
             total=torch.zeros(1, dtype=torch.int64, device="cuda"), overflow=torch.zeros(1, dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()      # torch's stream and the context's own stream are not ordered with each other
    return s


def run_shard_encode(c, x):
    """phases a..d of one rank that owns the whole image"""
    s = shard_buffers()
    dst = torch.empty(x.slot, dtype=torch.uint8, device="cuda")
    c.shard_encode_a(*(d[0] for d in x.dev), x.W, x.H, 0, x.VU, 0, False, s["last_dc"])
    c.shard_encode_b(s["dc_init"], s["info"])
    c.shard_encode_c(s["info"], 0, 1, s["nbytes"])
    c.shard_encode_d(s["nbytes"], dst, x.slot, s["total"], s["overflow"])


def run_decode(c, x):
    c.decode(x.scan0, x.frame)


def run_decode_batch(c, x):
    r, g, b = (np.zeros(NIMG * x.need, np.uint8) for _ in range(3))
    st = np.zeros(NIMG, np.int32)
    c.decode_batch(x.h_scan, x.slot, x.h_bytes, NIMG, x.frame, False, r, g, b, x.need, st)


def run_decode_batch_dev(c, x):
    c.decode_batch_dev(x.d_scan, x.slot, x.h_bytes, NIMG, x.frame, False, *x.planes_out(), x.need)


def run_decode_batch_dev2(c, x):
    c.decode_batch_dev2(x.d_scan, x.slot, x.d_bytes, int(x.h_bytes.max()), NIMG, x.frame, False, *x.planes_out(), x.need)


def run_shard_decode_dev(c, x):
    c.shard_decode_dev(x.d_scan[0], int(x.h_bytes[0]), x.frame, False, x.VU // 4, x.VU // 2, *x.planes_out(1), x.need)


def run_entropy_decode_dev(c, x):
    coefs = torch.empty((NIMG, x.nmcu * 384), dtype=torch.int16, device="cuda")
    c.entropy_decode_dev(x.d_scan, x.slot, x.h_bytes, NIMG, x.frame, coefs)


def run_transform_inv_dev(c, x):
    c.transform_inv_dev(x.coefs, x.frame, NIMG, False, *x.planes_out(), x.need)


RUNS = {f.__name__[4:]: f for f in (run_encode, run_encode_optimized, run_encode_batch, run_encode_batch_dev, run_encode_batch_optimized_dev,
                                    run_transform_fwd_dev, run_entropy_encode_dev, run_entropy_encode_optimized_dev, run_shard_encode,
                                    run_decode, run_decode_batch, run_decode_batch_dev, run_decode_batch_dev2, run_shard_decode_dev,
                                    run_entropy_decode_dev, run_transform_inv_dev)}

# kernel launches of (first call, second call) on a fresh context
LAUNCHES = {
    (512, 512): dict(encode=(8, 8), encode_optimized=(10, 10), encode_batch=(8, 8), encode_batch_dev=(8, 8), encode_batch_optimized_dev=(10, 10),
                transform_fwd_dev=(1, 1), entropy_encode_dev=(7, 7), entropy_encode_optimized_dev=(9, 9), shard_encode=(12, 12),
                decode=(14, 13), decode_batch=(14, 13), decode_batch_dev=(14, 13), decode_batch_dev2=(14, 13), shard_decode_dev=(14, 13),
                entropy_decode_dev=(12, 12), transform_inv_dev=(2, 1)),
    (1920, 1080): dict(encode=(8, 8), encode_optimized=(10, 10), encode_batch=(8, 8), encode_batch_dev=(8, 8), encode_batch_optimized_dev=(10, 10),
                    transform_fwd_dev=(1, 1), entropy_encode_dev=(7, 7), entropy_encode_optimized_dev=(9, 9), shard_encode=(12, 12),
                    decode=(14, 13), decode_batch=(14, 13), decode_batch_dev=(14, 13), decode_batch_dev2=(14, 13), shard_decode_dev=(14, 13),
                    entropy_decode_dev=(12, 12), transform_inv_dev=(2, 1)),
}


def launches(run, x):
    c = J.Context(0)
    try:
        got = []
        for _ in range(2):
            torch.cuda.synchronize()
            n0 = c.stat(capi.STAT_KERNEL_LAUNCHES)
            run(c, x)
            torch.cuda.synchronize()
            got.append(c.stat(capi.STAT_KERNEL_LAUNCHES) - n0)
        return tuple(got)
    finally:
        c.close()


@pytest.mark.parametrize("W,H", SIZES)
@pytest.mark.parametrize("entry", sorted(RUNS))
def test_kernel_launches(entry, W, H):
    got = launches(RUNS[entry], inputs(W, H))
    assert got == LAUNCHES[(W, H)].get(entry), "%s %dx%d launches %r" % (entry, W, H, got)


# ---- bad arguments ----------------------------------------------------------------------------------------------------
def _encode(c, x, h=True, r=True, W=None, H=None, cap=None, ht=True, fn="jpezyb200_encode"):
    cap = x.slot if cap is None else cap
    out = np.empty(max(cap, 1), np.uint8)
    n, nb, tabs = C.c_size_t(0), C.c_uint64(0), capi.HuffTables()
    args = [c.h if h else None, _dp(x.host[0][0]) if r else None, _dp(x.host[1][0]), _dp(x.host[2][0]), x.W if W is None else W,
            x.H if H is None else H, 0, _dp(out), cap, C.byref(n), C.byref(nb)]
    if fn == "jpezyb200_encode_optimized":
        args.append(C.byref(tabs) if ht else None)
    return getattr(c.lib, fn)(*args)


def _encode_opt(c, x, **kw):
    return _encode(c, x, fn="jpezyb200_encode_optimized", **kw)


def _encode_batch_dev(c, x, nimg=NIMG, slot=None, scan=True, ht=True, W=None, opt=False):
    out = torch.empty((NIMG, x.slot), dtype=torch.uint8, device="cuda")
    nb = torch.empty(NIMG, dtype=torch.int64, device="cuda")
    d_ht = torch.empty(NIMG * HB, dtype=torch.uint8, device="cuda")
    args = [c.h, *(_dp(d) for d in x.dev), x.W if W is None else W, x.H, nimg, 0, _dp(out) if scan else None,
            x.slot if slot is None else slot, _dp(nb), None]
    if opt:
        return c.lib.jpezyb200_encode_batch_optimized_dev(*args, _dp(d_ht) if ht else None, None)
    return c.lib.jpezyb200_encode_batch_dev(*args, None)


def _entropy_encode(c, x, coefs=True, slot=None, ht=True, opt=False):
    out = torch.empty((NIMG, x.slot), dtype=torch.uint8, device="cuda")
    nb = torch.empty(NIMG, dtype=torch.int64, device="cuda")
    d_ht = torch.empty(NIMG * HB, dtype=torch.uint8, device="cuda")
    args = [c.h, _dp(x.coefs) if coefs else None, x.W, x.H, NIMG, 0, _dp(out), x.slot if slot is None else slot, _dp(nb), None]
    if opt:
        return c.lib.jpezyb200_entropy_encode_optimized_dev(*args, _dp(d_ht) if ht else None, None)
    return c.lib.jpezyb200_entropy_encode_dev(*args, None)


def _transform_fwd(c, x, coefs=True):
    return c.lib.jpezyb200_transform_fwd_dev(c.h, *(_dp(d) for d in x.dev), x.W, x.H, NIMG, 0, _dp(x.coefs) if coefs else None, None)


def _read_sizes(c, x, n):
    out = np.zeros(max(n, 1), np.uint64)
    src = torch.empty(8200, dtype=torch.int64, device="cuda")
    return c.lib.jpezyb200_read_sizes(c.h, _dp(src), n, _dp(out), None)


def _frame(x, width=None):
    f = J.default_frame(x.W, x.H)
    if width is not None:
        f.width = width
    return f


def _decode(c, x, scan=True, n=None, plane=None, width=None):
    a = np.frombuffer(x.scan0, np.uint8)
    r, g, b = (np.zeros(x.need, np.uint8) for _ in range(3))
    f = _frame(x, width)
    return c.lib.jpezyb200_decode(c.h, _dp(a) if scan else None, a.size if n is None else n, C.byref(f), 0, _dp(r), _dp(g), _dp(b),
                                  x.need if plane is None else plane)


def _decode_batch_dev(c, x, bytes_=True, nimg=NIMG, lengths=None):
    hs = np.ascontiguousarray(x.h_bytes if lengths is None else lengths, dtype=np.uint64)
    return c.lib.jpezyb200_decode_batch_dev(c.h, _dp(x.d_scan), x.slot, _dp(hs) if bytes_ else None, nimg, C.byref(x.frame), 0,
                                            *(_dp(p) for p in x.planes_out()), x.need, None, None)


def _decode_batch_dev2(c, x, bytes_=True, nimg=NIMG, max_bytes=None):
    mx = int(x.h_bytes.max()) if max_bytes is None else max_bytes
    return c.lib.jpezyb200_decode_batch_dev2(c.h, _dp(x.d_scan), x.slot, _dp(x.d_bytes) if bytes_ else None, mx, nimg, C.byref(x.frame),
                                             0, *(_dp(p) for p in x.planes_out()), x.need, None, None)


def _entropy_decode(c, x, coefs=True):
    d = torch.empty((NIMG, x.nmcu * 384), dtype=torch.int16, device="cuda")
    hs = np.ascontiguousarray(x.h_bytes)
    return c.lib.jpezyb200_entropy_decode_dev(c.h, _dp(x.d_scan), x.slot, _dp(hs), NIMG, C.byref(x.frame), _dp(d) if coefs else None,
                                              None, None)


def _transform_inv(c, x, plane=None):
    return c.lib.jpezyb200_transform_inv_dev(c.h, _dp(x.coefs), C.byref(x.frame), NIMG, 0, *(_dp(p) for p in x.planes_out()),
                                             x.need if plane is None else plane, None)


def _shard_decode(c, x, row0, rows, n=None):
    return c.lib.jpezyb200_shard_decode_dev(c.h, _dp(x.d_scan[0]), int(x.h_bytes[0]) if n is None else n, C.byref(x.frame), 0, row0,
                                            rows, *(_dp(p) for p in x.planes_out(1)), x.need, None, None)


def _shard_phases(c, x, order, row0=0, rows=None, y_origin=0):
    """runs the shard phases named in `order` ("a".."d") and returns the status of the last; the earlier ones must succeed"""
    s = shard_buffers()
    dst = torch.empty(x.slot, dtype=torch.uint8, device="cuda")
    rows = x.VU if rows is None else rows
    calls = {
        "a": lambda: c.lib.jpezyb200_shard_encode_a(c.h, *(_dp(d[0]) for d in x.dev), x.W, x.H, row0, rows, y_origin, 0, _dp(s["last_dc"]), None),
        "b": lambda: c.lib.jpezyb200_shard_encode_b(c.h, _dp(s["dc_init"]), _dp(s["info"]), None),
        "c": lambda: c.lib.jpezyb200_shard_encode_c(c.h, _dp(s["info"]), 0, 1, _dp(s["nbytes"]), None),
        "d": lambda: c.lib.jpezyb200_shard_encode_d(c.h, _dp(s["nbytes"]), _dp(dst), x.slot, _dp(s["total"]), _dp(s["overflow"]), None),
    }
    for k in order[:-1]:
        assert calls[k]() == OK, k
    return calls[order[-1]]()


def _encode_batch(c, x, slot=None):
    out = np.empty(NIMG * x.slot, np.uint8)
    nb = np.zeros(NIMG, np.uint64)
    return c.lib.jpezyb200_encode_batch(c.h, *(_dp(a) for a in x.host), x.W, x.H, NIMG, 0, _dp(out), x.slot if slot is None else slot,
                                        _dp(nb))


def _decode_batch(c, x, lengths=None):
    hs = np.ascontiguousarray(x.h_bytes if lengths is None else lengths, dtype=np.uint64)
    r, g, b = (np.zeros(NIMG * x.need, np.uint8) for _ in range(3))
    return c.lib.jpezyb200_decode_batch(c.h, _dp(x.h_scan), x.slot, _dp(hs), NIMG, C.byref(x.frame), 0, _dp(r), _dp(g), _dp(b), x.need, None)


BAD = {
    "encode/null ctx": (lambda c, x: _encode(c, x, h=False), EINVAL),
    "encode/null r": (lambda c, x: _encode(c, x, r=False), EINVAL),
    "encode/zero cap": (lambda c, x: _encode(c, x, cap=0), EINVAL),
    "encode/width 65536": (lambda c, x: _encode(c, x, W=65536), EINVAL),
    "encode/height 0": (lambda c, x: _encode(c, x, H=0), EINVAL),
    "encode/cap 64": (lambda c, x: _encode(c, x, cap=64), ECAPACITY),
    "encode_optimized/null ctx": (lambda c, x: _encode_opt(c, x, h=False), EINVAL),
    "encode_optimized/null ht": (lambda c, x: _encode_opt(c, x, ht=False), EINVAL),
    "encode_optimized/zero cap": (lambda c, x: _encode_opt(c, x, cap=0), EINVAL),
    "encode_optimized/height 65536": (lambda c, x: _encode_opt(c, x, H=65536), EINVAL),
    "encode_optimized/cap 64": (lambda c, x: _encode_opt(c, x, cap=64), ECAPACITY),
    "encode_batch_dev/nimg 0": (lambda c, x: _encode_batch_dev(c, x, nimg=0), EINVAL),
    "encode_batch_dev/nimg 65536": (lambda c, x: _encode_batch_dev(c, x, nimg=65536), EINVAL),
    "encode_batch_dev/zero slot": (lambda c, x: _encode_batch_dev(c, x, slot=0), EINVAL),
    "encode_batch_dev/null scan": (lambda c, x: _encode_batch_dev(c, x, scan=False), EINVAL),
    "encode_batch_dev/width 65536": (lambda c, x: _encode_batch_dev(c, x, W=65536), EINVAL),
    "encode_batch_optimized_dev/null ht": (lambda c, x: _encode_batch_dev(c, x, opt=True, ht=False), EINVAL),
    "encode_batch_optimized_dev/zero slot": (lambda c, x: _encode_batch_dev(c, x, opt=True, slot=0), EINVAL),
    "encode_batch_optimized_dev/nimg 0": (lambda c, x: _encode_batch_dev(c, x, opt=True, nimg=0), EINVAL),
    "entropy_encode_dev/null coefs": (lambda c, x: _entropy_encode(c, x, coefs=False), EINVAL),
    "entropy_encode_dev/zero slot": (lambda c, x: _entropy_encode(c, x, slot=0), EINVAL),
    "entropy_encode_optimized_dev/null ht": (lambda c, x: _entropy_encode(c, x, opt=True, ht=False), EINVAL),
    "entropy_encode_optimized_dev/null coefs": (lambda c, x: _entropy_encode(c, x, opt=True, coefs=False), EINVAL),
    "transform_fwd_dev/null coefs": (lambda c, x: _transform_fwd(c, x, coefs=False), EINVAL),
    "read_sizes/n 0": (lambda c, x: _read_sizes(c, x, 0), EINVAL),
    "read_sizes/n 8193": (lambda c, x: _read_sizes(c, x, 8193), EINVAL),
    "encode_batch/zero slot": (lambda c, x: _encode_batch(c, x, slot=0), EINVAL),
    "decode/null scan": (lambda c, x: _decode(c, x, scan=False), EINVAL),
    "decode/zero bytes": (lambda c, x: _decode(c, x, n=0), EINVAL),
    "decode/planes too small": (lambda c, x: _decode(c, x, plane=x.need - 1), ECAPACITY),
    "decode/width 65536": (lambda c, x: _decode(c, x, width=65536), EINVAL),
    "decode_batch/zero length": (lambda c, x: _decode_batch(c, x, lengths=[0] * NIMG), EINVAL),
    "decode_batch_dev/null lengths": (lambda c, x: _decode_batch_dev(c, x, bytes_=False), EINVAL),
    "decode_batch_dev/nimg 0": (lambda c, x: _decode_batch_dev(c, x, nimg=0), EINVAL),
    "decode_batch_dev/length above slot": (lambda c, x: _decode_batch_dev(c, x, lengths=[x.slot + 1] * NIMG), EINVAL),
    "decode_batch_dev/zero lengths": (lambda c, x: _decode_batch_dev(c, x, lengths=[0] * NIMG), ECORRUPT),
    "decode_batch_dev2/null lengths": (lambda c, x: _decode_batch_dev2(c, x, bytes_=False), EINVAL),
    "decode_batch_dev2/nimg 0": (lambda c, x: _decode_batch_dev2(c, x, nimg=0), EINVAL),
    "decode_batch_dev2/max 0": (lambda c, x: _decode_batch_dev2(c, x, max_bytes=0), EINVAL),
    "decode_batch_dev2/max above slot": (lambda c, x: _decode_batch_dev2(c, x, max_bytes=x.slot + 1), EINVAL),
    "entropy_decode_dev/null coefs": (lambda c, x: _entropy_decode(c, x, coefs=False), EINVAL),
    "transform_inv_dev/planes too small": (lambda c, x: _transform_inv(c, x, plane=x.need - 1), ECAPACITY),
    "shard_decode_dev/zero rows": (lambda c, x: _shard_decode(c, x, 0, 0), EINVAL),
    "shard_decode_dev/row0 past the image": (lambda c, x: _shard_decode(c, x, x.VU, 1), EINVAL),
    "shard_decode_dev/rows past the image": (lambda c, x: _shard_decode(c, x, 1, x.VU), EINVAL),
    "shard_decode_dev/zero bytes": (lambda c, x: _shard_decode(c, x, 0, 1, n=0), EINVAL),
    "shard_encode_a/rows past the image": (lambda c, x: _shard_phases(c, x, "a", row0=1, rows=x.VU), EINVAL),
    "shard_encode_a/y_origin below the shard": (lambda c, x: _shard_phases(c, x, "a", row0=1, rows=1, y_origin=17), EINVAL),
    "shard_encode/b first": (lambda c, x: _shard_phases(c, x, "b"), EINVAL),
    "shard_encode/c first": (lambda c, x: _shard_phases(c, x, "c"), EINVAL),
    "shard_encode/d first": (lambda c, x: _shard_phases(c, x, "d"), EINVAL),
    "shard_encode/c after a": (lambda c, x: _shard_phases(c, x, "ac"), EINVAL),
    "shard_encode/d after a": (lambda c, x: _shard_phases(c, x, "ad"), EINVAL),
    "shard_encode/d after b": (lambda c, x: _shard_phases(c, x, "abd"), EINVAL),
    "shard_encode/b twice": (lambda c, x: _shard_phases(c, x, "abb"), EINVAL),
    "shard_encode/b after d": (lambda c, x: _shard_phases(c, x, "abcdb"), EINVAL),
    "shard_encode/a..d": (lambda c, x: _shard_phases(c, x, "abcd"), OK),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_bad_arguments(case):
    call, want = BAD[case]
    x = inputs(*SIZES[0])
    c = J.Context(0)
    try:
        torch.cuda.synchronize()
        got = call(c, x)
        torch.cuda.synchronize()
    finally:
        c.close()
    assert got == want, "%s: status %d" % (case, got)
