"""Test-side pixel builder for the forward transform (numpy only): it proposes RGB pixels whose colour-converted samples hit
chosen DCT values, and certifies what those pixels do from the reference's own FP64 DCT values (oracle.coefs(...,
want_raw=True)), so no test relies on the builder's arithmetic.

- Luma: a pixel with Cb = Cr = 0 is found for every Y sample (gray where the reference's FP64 rounding allows it).
- Chroma: the samples come from the even/even pixel of each 2x2; an inverse of the reference's colour formulas (evaluated
  as the reference evaluates them) writes any Cb sample with Cr = 0 and any Cr sample with Cb = 0 (|sample| <= 120).
- Certificate: every AC coefficient's distance to the nearest non-zero multiple of its quantiser, in units of the guard band
  G that k_fwd_transform uses (G = (1.25 kAanErrBound[i][j] + 5e-4) / q, jpezy_b200/csrc/capi.cu, with the bound table
  parsed out of enc_transform.cuh).  The FP32 flowgraph's error is at most kAanErrBound / q, so a coefficient is certainly
  queued below 1 - B/(qG) and certainly not queued above 1 + B/(qG).

Sample blocks are 8x8 int arrays in natural order; `Canvas` places them into MCUs (Y0 Y1 Y2 Y3 Cb Cr) of an image.

Families: exact quantisation ties (ties_image); 32-MCU tiles with 1023, 1024, 1025 and 1152 coefficients certainly in the
kernel's fix-up queue of 1024 entries (queue_image); blocks at chosen distances from the guard band at every AC position of
both classes (sweep_image); every zig-zag group mask of the entropy coders' side information with all-black, all-white and
DC-only blocks (mask_image); ragged frames (ragged_image)."""
import functools
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# T.81 Annex K tables K.1 / K.2, natural order (jpezy_b200/csrc/tables.h)
QY = np.array([16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
               14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92,
               49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99], np.int64)
QC = np.array([17, 18, 24, 47] + [99] * 4 + [18, 21, 26, 66] + [99] * 4 + [24, 26, 56] + [99] * 5 + [47, 66] + [99] * 38,
              np.int64)
Q = np.stack([QY, QC])
ZZ = np.array(sorted(range(64), key=lambda n: (n // 8 + n % 8, (n // 8) if (n // 8 + n % 8) % 2 else -(n // 8))))   # zig-zag -> natural
_u = np.arange(8)
COS = np.cos((2 * _u[None, :] + 1) * _u[:, None] * np.pi / 16)          # COS[u][x]
_CU = np.where(_u == 0, 2 ** -0.5, 1.0)
LUMA_RANGE, CHROMA_RANGE = (-128, 127), (-120, 120)


def basis(i, j):
    """8x8 weights: F(i, j) = sum(basis * samples)"""
    return np.outer(COS[i], COS[j]) * _CU[i] * _CU[j] / 4


def dct(s):
    """[..., 8, 8] samples -> [..., 8, 8] DCT in the reference's scaling (float64; the oracle's values certify)"""
    return np.einsum("iy,...yx,jx->...ij", COS, np.asarray(s, np.float64), COS) * np.outer(_CU, _CU) / 4


def idct(F):
    return np.einsum("iy,...ij,jx->...yx", COS, np.asarray(F, np.float64) * np.outer(_CU, _CU) / 4, COS)


def quantise(F, cls):
    """the reference's int(v) / q, natural order"""
    return np.fix(np.trunc(np.asarray(F)).reshape(-1, 64) / Q[cls]).astype(np.int64)


# ---- the kernel's guard band -----------------------------------------------------------------------------------------
@functools.lru_cache(None)
def aan_err_bound():
    """kAanErrBound[64] as written in jpezy_b200/csrc/enc_transform.cuh"""
    src = open(os.path.join(ROOT, "jpezy_b200", "csrc", "enc_transform.cuh")).read()
    body = re.search(r"kAanErrBound\[64\]\s*=\s*\{([^}]*)\}", src).group(1)
    vals = np.array([float(x.strip().rstrip("f")) for x in body.split(",") if x.strip()])
    assert vals.shape == (64,)
    return vals


def guard():
    """[class][64] guard band G in w = v / q units, as capi.cu computes it (in double; the kernel holds it as float)"""
    return (1.25 * aan_err_bound()[None, :] + 5e-4) / Q


def certify(raw, gray=False):
    """raw: oracle raw DCT values [nmcu, 6, 64] (natural order) -> distance of every coefficient to the nearest non-zero
    multiple of q, in units of G (DC: inf)"""
    raw = np.asarray(raw, np.float64).reshape(-1, 6, 64)
    cls = (np.arange(6) >= 4).astype(np.int64)
    w = np.abs(raw) / Q[cls][None]
    d = np.abs(w - np.maximum(1.0, np.round(w))) / guard()[cls][None]
    d[:, :, 0] = np.inf
    return d


def queue_limits():
    """[class][64] (certainly queued below, certainly not queued above), in units of G"""
    e = aan_err_bound()[None, :] / Q / guard()
    return 1.0 - e, 1.0 + e


def queued(dist):
    """-> (certainly queued, uncertain) boolean arrays of a certify() result"""
    lo, hi = queue_limits()
    cls = (np.arange(6) >= 4).astype(np.int64)
    lo, hi = lo[cls][None], hi[cls][None]
    return dist < lo, (dist >= lo) & (dist <= hi)


# ---- colour ------------------------------------------------------------------------------------------------------------
def ref_y(r, g, b):
    r, g, b = (np.asarray(x, np.float64) for x in (r, g, b))
    return np.trunc((0.2990 * r + 0.5870 * g) + 0.1140 * b - 128).astype(np.int64)


def ref_cb(r, g, b):
    r, g, b = (np.asarray(x, np.float64) for x in (r, g, b))
    return np.trunc((-(0.1687 * r) - 0.3313 * g) + 0.5000 * b).astype(np.int64)


def ref_cr(r, g, b):
    r, g, b = (np.asarray(x, np.float64) for x in (r, g, b))
    return np.trunc((0.5000 * r - 0.4187 * g) - 0.0813 * b).astype(np.int64)


@functools.lru_cache(None)
def colour_tables():
    """-> (luma[256], cb[241], cr[241], pair[256 * 256]): packed 0xRRGGBB pixels giving Y = s with Cb = Cr = 0 (index s + 128),
    Cb = s with Cr = 0 and Cr = s with Cb = 0 (index s + 120), and (Cb, Cr) (index (Cb + 128) * 256 + Cr + 128; -1: none);
    gray pixels where they do it"""
    v = np.arange(256, dtype=np.float64)
    g, b = np.meshgrid(v, v, indexing="ij")
    gb = (g.astype(np.int64) << 8) | b.astype(np.int64)
    luma, cb, cr = np.full(256, -1, np.int64), np.full(241, -1, np.int64), np.full(241, -1, np.int64)
    pair = np.full(65536, -1, np.int64)
    for r in range(256):
        y, u, w = ref_y(r, g, b), ref_cb(r, g, b), ref_cr(r, g, b)
        pix = (r << 16) | gb
        for tbl, m, key in ((luma, (u == 0) & (w == 0), y + 128), (cb, w == 0, u + 120), (cr, u == 0, w + 120),
                             (pair, u == u, (u + 128) * 256 + w + 128)):
            m = m & (key >= 0) & (key < tbl.size)
            k, p = key[m], pix[m]
            free = tbl[k] < 0
            tbl[k[free]] = p[free]
    gray = ref_y(v, v, v) + 128
    ok = (ref_cb(v, v, v) == 0) & (ref_cr(v, v, v) == 0)
    luma[gray[ok]] = (np.arange(256)[ok] * 0x010101)
    assert (luma >= 0).all() and (cb >= 0).all() and (cr >= 0).all()
    return luma, cb, cr, pair


def unpack(p):
    p = np.asarray(p, np.int64)
    return ((p >> 16) & 255).astype(np.uint8), ((p >> 8) & 255).astype(np.uint8), (p & 255).astype(np.uint8)


class Canvas:
    """HU x VU MCUs of pixels; luma(m, k, s) writes luma block k of MCU m (its chroma stays 0 where chroma() did not write),
    chroma(m, c, s) writes the Cb (c = 0) or Cr (c = 1) block of MCU m (the other one 0; the luma of the even/even pixels
    follows, the other pixels stay as they are)"""

    def __init__(self, HU, VU, fill=128):
        self.HU, self.VU = HU, VU
        self.W, self.H = HU * 16, VU * 16
        self.pix = np.full((self.H, self.W), fill * 0x010101, np.int64)

    def _mcu(self, m):
        return (m // self.HU) * 16, (m % self.HU) * 16

    def luma(self, m, k, s):
        s = np.asarray(s, np.int64).reshape(8, 8)
        assert s.min() >= LUMA_RANGE[0] and s.max() <= LUMA_RANGE[1]
        y0, x0 = self._mcu(m)
        y0, x0 = y0 + (k >> 1) * 8, x0 + (k & 1) * 8
        self.pix[y0:y0 + 8, x0:x0 + 8] = colour_tables()[0][s + 128]

    def chroma(self, m, c, s):
        s = np.asarray(s, np.int64).reshape(8, 8)
        assert s.min() >= CHROMA_RANGE[0] and s.max() <= CHROMA_RANGE[1]
        y0, x0 = self._mcu(m)
        self.pix[y0:y0 + 16:2, x0:x0 + 16:2] = colour_tables()[1 + c][s + 120]

    def chroma2(self, m, cb, cr):
        """both chroma blocks of MCU m (|samples| <= PAIR_RANGE)"""
        cb, cr = (np.asarray(x, np.int64).reshape(8, 8) for x in (cb, cr))
        p = colour_tables()[3][(cb + 128) * 256 + cr + 128]
        assert (p >= 0).all()
        y0, x0 = self._mcu(m)
        self.pix[y0:y0 + 16:2, x0:x0 + 16:2] = p

    def planes(self, W=None, H=None):
        W, H = W or self.W, H or self.H
        return unpack(self.pix[:H, :W])


# ---- blocks --------------------------------------------------------------------------------------------------------------
def _types():
    """pixel orbits under y -> 7 - y, x -> 7 - x (16 types of 4 pixels): the even/even coefficients depend only on the sums
    of the samples over each orbit"""
    t = np.minimum(_u, 7 - _u)
    return (t[:, None] * 4 + t[None, :]).reshape(-1)


TYPES = _types()
RATIONAL = [(0, 4), (4, 0), (4, 4)]          # values are multiples of 1/8 for any integer block
SQRT2 = [(2, 2), (2, 6), (6, 2), (6, 6)]      # values lie in Q(sqrt 2)
# Over the 16 orbit sums the forms of the SQRT2 positions span four dimensions: once every value is rational,
# F(2,2) = F(6,6) and F(2,6) = -F(6,2).  Both members of a pair tie only when their quantisers allow the same value: in luma
# (q 16 and 120) at F(2,2) = F(6,6) = 240 k, in chroma (q 99 and 99) at F(2,6) = -F(6,2) = 99 k.  Six ties per block:
TIE6 = [[RATIONAL + [(2, 2), (6, 6), (2, 6)], RATIONAL + [(2, 2), (6, 6), (6, 2)]],         # luma
        [RATIONAL + [(2, 2), (2, 6), (6, 2)], RATIONAL + [(6, 6), (2, 6), (6, 2)]]]         # chroma
# luma blocks with exactly five and four ties (F(6,2) = -69 k * q26 / q62 and F(6,6) = F(2,2) are not multiples of q there)
TIE5_LUMA = [RATIONAL + [(2, 2), (2, 6)], RATIONAL + [(6, 2), (6, 6)]]
TIE4_LUMA = [RATIONAL + [(2, 6)], RATIONAL + [(6, 2)]]
TIE_SETS = TIE5_LUMA


def tie_ks(rng, positions, cls, mag=1):
    """multiples k of q for the positions of a tie set: the pair constraints of TIE6 respected, |k| = mag where q < 70"""
    ks = {p: (mag if Q[cls][p[0] * 8 + p[1]] < 70 else 1) * (1 if rng.random() < 0.5 else -1) for p in positions}
    if (2, 2) in ks and (6, 6) in ks:
        assert cls == 0
        sg = 1 if rng.random() < 0.5 else -1
        ks[(2, 2)], ks[(6, 6)] = sg * 15, sg * 2
    if (2, 6) in ks and (6, 2) in ks:
        ks[(6, 2)] = -ks[(2, 6)] * int(Q[cls][22]) // int(Q[cls][50])
    return [ks[p] for p in positions]


def tie_forms(i, j):
    """integer forms over the 64 samples and their targets for F(i, j) = k q: [(form, scale)] with sum(form * s) = scale * k * q"""
    if (i, j) in RATIONAL:          # F = sum(+-s) / 8
        return [(np.outer(np.sign(np.round(COS[i] * 8)), np.sign(np.round(COS[j] * 8))).reshape(-1).astype(np.int64), 8)]
    a = np.isclose(np.abs(COS[i]), np.cos(np.pi / 8))[:, None], np.isclose(np.abs(COS[j]), np.cos(np.pi / 8))[None, :]
    sg = np.outer(np.sign(COS[i]), np.sign(COS[j]))
    aa, bb = a[0] & a[1], ~a[0] & ~a[1]
    # c_i(y) c_j(x) = (r + t sqrt 2) / 4 with (r, t) = (2, 1) on a*a, (2, -1) on b*b, (0, 1) on a*b: F = (sum r s + sqrt 2 sum t s) / 16
    t = (np.where(aa, 1, np.where(bb, -1, 1)) * sg).reshape(-1).astype(np.int64)
    r2 = (np.where(aa | bb, 1, 0) * sg).reshape(-1).astype(np.int64)
    return [(t, 0), (r2, 8)]


def _greedy(M, t, x, lo, hi, rng, iters=300):
    """integer x in [lo, hi] with M x = t by single and pair +-1 steps from x; None when it gets stuck"""
    x = x.copy()
    n = x.size
    lo, hi = np.broadcast_to(lo, (n,)), np.broadcast_to(hi, (n,))
    for _ in range(iters):
        r = t - M @ x
        n0 = np.abs(r).sum()
        if n0 == 0:
            return x
        best = (n0, None)
        for d1 in (1, -1):
            ok1 = (x + d1 >= lo) & (x + d1 <= hi)
            sc = np.abs(r[:, None] - d1 * M).sum(0) + np.where(ok1, 0, 1 << 40) + rng.random(n) * 0.1
            p = int(np.argmin(sc))
            if sc[p] < best[0]:
                best = (sc[p], [(p, d1)])
            for d2 in (1, -1):
                ok2 = (x + d2 >= lo) & (x + d2 <= hi)
                R = r[:, None, None] - d1 * M[:, :, None] - d2 * M[:, None, :]
                sc = np.abs(R).sum(0) + np.where(ok1[:, None] & ok2[None, :], 0, 1 << 40) + np.eye(n) * (1 << 40) + rng.random((n, n)) * 0.1
                k = int(np.argmin(sc))
                if sc.flat[k] < best[0]:
                    best = (sc.flat[k], [(k // n, d1), (k % n, d2)])
        if best[1] is None:
            p = int(rng.integers(n))
            x[p] = np.clip(x[p] + rng.choice([-1, 1]), lo[p], hi[p])
            continue
        for p, d in best[1]:
            x[p] += d
    return None


def tie_block(rng, positions, ks, cls, lo, hi, base=None, fixed=None):
    """integer samples in [lo, hi] whose exact DCT value at every positions[n] is ks[n] * q (a quantisation tie); solved on
    the 16 orbit sums, then spread over the orbits' pixels at random.  fixed: 8x8 samples that must stay (others: any value
    outside [lo, hi]), at most one per orbit.  None when the search fails."""
    M, t = [], []
    for (i, j), k in zip(positions, ks):
        for f, sc in tie_forms(i, j):
            M.append(np.array([f[TYPES == T][0] for T in range(16)]))
            t.append(sc * int(k) * int(Q[cls][i * 8 + j]))
    M, t = np.array(M), np.array(t)
    base = rng.integers(lo // 2, hi // 2 + 1, 64) if base is None else np.asarray(base, np.int64).reshape(-1)
    fx = np.full(64, hi + 1, np.int64) if fixed is None else np.asarray(fixed, np.int64).reshape(-1)
    isf = (fx >= lo) & (fx <= hi)
    nfree = np.array([4 - isf[TYPES == T].sum() for T in range(16)])
    fsum = np.array([fx[(TYPES == T) & isf].sum() for T in range(16)])
    assert (nfree >= 3).all()
    slo, shi = fsum + nfree * lo, fsum + nfree * hi
    sums = np.array([base[TYPES == T].sum() for T in range(16)])
    d = np.linalg.lstsq(M.astype(np.float64), (t - M @ sums).astype(np.float64), rcond=None)[0]
    sums = np.clip(sums + np.round(d).astype(np.int64), slo, shi)
    sums = _greedy(M, t, sums, slo, shi, rng)
    if sums is None:
        return None
    s = fx.copy()
    for T in range(16):
        idx = np.nonzero((TYPES == T) & ~isf)[0]
        n, rest = len(idx), sums[T] - fsum[T]
        part = np.full(n, rest // n) + (np.arange(n) < rest % n)
        for _ in range(6):        # texture: moves inside the orbit keep every even/even coefficient
            a, b = rng.choice(n, 2, replace=False)
            m = int(rng.integers(0, 1 + min(part[a] - lo, hi - part[b])))
            part[a] -= m
            part[b] += m
        s[idx] = part
    return s.reshape(8, 8)


def mask_block(rng, mask, cls, lo, hi, tries=200):
    """samples whose quantised AC coefficients are non-zero in exactly the zig-zag groups of `mask` (group g: zig-zag
    g*8 .. g*8+7, group 0 without the DC): one coefficient per chosen group at 1.5 q, inverse DCT, rounding"""
    for _ in range(tries):
        F = np.zeros(64)
        for g in range(8):
            if mask >> g & 1:
                z = int(rng.integers(max(1, 8 * g), 8 * g + 8))
                n = ZZ[z]
                F[n] = rng.choice([-1.5, 1.5]) * Q[cls][n]
        F[0] = rng.integers(-200, 200)
        s = np.round(idct(F.reshape(8, 8))).astype(np.int64)
        if s.min() < lo or s.max() > hi:
            continue
        qz = quantise(dct(s), cls)[0][ZZ]
        got = sum(1 << g for g in range(8) if qz[max(1, 8 * g):8 * g + 8].any())
        if got == mask:
            return s
    return None


PAIR_RANGE = (-80, 80)


# ---- families ------------------------------------------------------------------------------------------------------------
def ties_image(seed, HU=8, VU=2):
    """exact ties at the seven reachable positions in luma, Cb and Cr, both signs, k = +-1 and, where q < 70, |k| = 2, 3; every
    tie block solves one of TIE_SETS (five ties in luma; six in chroma, where F(6,2) = -F(2,6) and q is 99 at both).  A pixel fixes Y, Cb and Cr at once, so even MCUs carry four luma tie blocks (chroma
    0) and odd MCUs a Cb and a Cr tie block (their luma follows from the chroma pixels).  -> (r, g, b, W, H)"""
    rng = np.random.default_rng(seed)
    cv = Canvas(HU, VU)

    def solve(big, set_idx, cls, lo, hi):
        while True:
            mag = int(rng.integers(2, 4)) if big else 1
            pos = TIE_SETS[set_idx]
            ks = [(mag if Q[cls][i * 8 + j] < 70 else 1) * (1 if rng.random() < 0.5 else -1) for i, j in pos]
            s = tie_block(rng, pos, ks, cls, lo, hi)
            if s is not None:
                return s

    for m in range(HU * VU):
        if m % 2 == 0:
            for k in range(4):
                cv.luma(m, k, solve(k & 1, k >> 1, 0, *LUMA_RANGE))
        else:
            big = (m >> 2) & 1
            cv.chroma2(m, solve(big, (m >> 1) & 1, 1, *PAIR_RANGE), solve(1 - big, (m >> 1) & 1, 1, *PAIR_RANGE))
    return cv.planes() + (cv.W, cv.H)


def mask_image(seed, HU=32):
    """blocks whose quantised AC coefficients are non-zero in exactly the zig-zag groups of each of the 256 masks, in luma, Cb
    and Cr; then all-black and all-white MCUs and DC-only blocks over the whole DC range.  -> (r, g, b, W, H)"""
    rng = np.random.default_rng(seed)
    luma = [mask_block(rng, m, 0, *LUMA_RANGE) for m in range(256)]
    chroma = [mask_block(rng, m, 1, *CHROMA_RANGE) for m in range(256)]
    assert all(x is not None for x in luma + chroma)
    dc = [np.full((8, 8), v, np.int64) for v in range(-128, 128, 3)]
    nm = 64 + 256 + 2 + -(-len(dc) // 4)
    cv = Canvas(HU, -(-nm // HU))
    for e, s in enumerate(luma):
        cv.luma(e // 4, e % 4, s)
    for e, s in enumerate(chroma):
        cv.chroma(64 + e, e % 2, s)
    m = 64 + 256
    cv.pix[(m // HU) * 16:(m // HU) * 16 + 16, (m % HU) * 16:(m % HU) * 16 + 16] = 0
    m += 1
    cv.pix[(m // HU) * 16:(m // HU) * 16 + 16, (m % HU) * 16:(m % HU) * 16 + 16] = 0xFFFFFF
    for e, s in enumerate(dc):
        cv.luma(m + 1 + e // 4, e % 4, s)
    return cv.planes() + (cv.W, cv.H)


def ragged_image(seed, W, H):
    """smooth random content with 0/255 alternation in the last column and the last row (edge replication copies them across
    the rest of the MCU) -> (r, g, b)"""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:H, 0:W]
    planes = []
    for c in range(3):
        f = rng.uniform(0.02, 0.3, 2)
        p = 128 + 100 * np.sin(f[0] * x + rng.uniform(0, 6)) * np.cos(f[1] * y) + rng.normal(0, 12, (H, W))
        p = np.clip(np.round(p), 0, 255).astype(np.uint8)
        p[:, W - 1] = np.where(np.arange(H) % 2, 255, 0)
        p[H - 1, :] = np.where(np.arange(W) % 2, 0, 255)
        planes.append(np.ascontiguousarray(p))
    return tuple(planes)


def _only(s, cls, positions):
    """every AC coefficient of s outside `positions` certainly stays out of the guard-band queue (builder-side, float64)"""
    d = np.abs(dct(s)).reshape(64) / Q[cls]
    d = np.abs(d - np.maximum(1.0, np.round(d))) / guard()[cls]
    d[[0] + [i * 8 + j for i, j in positions]] = np.inf
    return (d > queue_limits()[1][cls] + 0.5).all()


def _tie(rng, sets, cls, lo, hi, fixed=None, tries=400):
    for n in range(tries):
        pos = sets[n % len(sets)]
        s = tie_block(rng, pos, tie_ks(rng, pos, cls), cls, lo, hi, fixed=fixed)
        if s is not None and _only(s, cls, pos):
            return s
    raise RuntimeError("no tie block found")


QUEUE_COUNTS = (1023, 1024, 1025, 1152)


def queue_image(seed, counts=QUEUE_COUNTS):
    """one 32-MCU tile of k_fwd_transform (512 x 16 pixels) per entry of `counts`, each with exactly that many exact ties
    and no other AC coefficient near the guard band: Cb and Cr blocks hold six ties each (TIE6), the 128 luma blocks four,
    five or six.  Luma and chroma share the MCUs: the chroma pixels (one per orbit of every luma block) are placed first and
    the luma ties are solved around their Y values.  -> (r, g, b, W, H)"""
    rng = np.random.default_rng(seed)
    cv = Canvas(32, len(counts))
    luma_t = colour_tables()[3]
    for row, count in enumerate(counts):
        nl = count - 64 * 6                                  # luma ties of the tile
        per = [5] * 128
        for b in range(abs(nl - 640)):
            per[b * 13 % 128] = 6 if nl > 640 else 4
        assert sum(per) == nl and set(per) <= {4, 5, 6}
        for mx in range(32):
            m = row * 32 + mx
            cb = _tie(rng, TIE6[1], 1, *PAIR_RANGE)
            cr = _tie(rng, TIE6[1], 1, *PAIR_RANGE)
            cv.chroma2(m, cb, cr)
            y_ee = ref_y(*unpack(luma_t[(cb + 128) * 256 + cr + 128]))       # Y of the 8x8 even/even pixels of the MCU
            for k in range(4):
                fixed = np.full((8, 8), 1 << 20, np.int64)
                fixed[0::2, 0::2] = y_ee[(k >> 1) * 4:(k >> 1) * 4 + 4, (k & 1) * 4:(k & 1) * 4 + 4]
                sets = {4: TIE4_LUMA, 5: TIE5_LUMA, 6: TIE6[0]}[per[mx * 4 + k]]
                s = _tie(rng, sets, 0, *LUMA_RANGE, fixed=fixed)
                y0, x0 = cv._mcu(m)
                y0, x0 = y0 + (k >> 1) * 8, x0 + (k & 1) * 8
                odd = np.ones((8, 8), bool)
                odd[0::2, 0::2] = False
                cv.pix[y0:y0 + 8, x0:x0 + 8][odd] = colour_tables()[0][s[odd] + 128]
    return cv.planes() + (cv.W, cv.H)


SWEEP = (0.1, 0.5, 1.0, 2.0, 4.0)            # distances from k q in units of G, on alternating sides, k = |w| - 1 of the block
SWEEP_T = (-2.5, -1.5, -0.5, 0.5)           # around |w| = 1, where the kernel's "quantises to 0" skip (|w| < 1 - 2G) decides


def sweep_block(rng, cls, i, j, k, delta, R, tries=300):
    """samples in [-R, R] with F(i, j) = (k + delta G) q within 0.08 G q, k = None: the k at 60 % of the value of the
    position's +-R sign pattern (high contrast).  F is sum over magnitude groups m_g T_g (T_g: signed sample sum of the
    pixels of weight +-m_g): all but two groups are set near a common fraction of their range, the pair is enumerated."""
    n = i * 8 + j
    q, G = float(Q[cls][n]), float(guard()[cls][n])
    B = basis(i, j).reshape(64)
    mag = np.round(np.abs(B), 12)
    groups = [np.nonzero(mag == m)[0] for m in np.unique(mag)]
    m = np.array([abs(B[g[0]]) for g in groups])
    cnt = np.array([len(g) for g in groups])
    vmax = R * float((m * cnt).sum())
    if k is None:
        k = max(1, int(0.6 * vmax / q))     # (room for the enumerated pair)
    target, tol = (k + delta * G) * q, 0.08 * G * q
    assert 0 < target < vmax
    for _ in range(tries):
        f = np.clip(target / vmax + rng.normal(0, 0.05, len(groups)), -1, 1)
        T = np.round(f * cnt * R).astype(np.int64)
        g1, g2 = rng.choice(len(groups), 2, replace=False)
        rest = target - float((m * T).sum()) + m[g1] * T[g1] + m[g2] * T[g2]
        t1 = np.arange(-cnt[g1] * R, cnt[g1] * R + 1)
        t2 = np.round((rest - m[g1] * t1) / m[g2]).astype(np.int64)
        err = np.abs(m[g1] * t1 + m[g2] * t2 - rest)
        ok = np.nonzero((np.abs(t2) <= cnt[g2] * R) & (err < tol))[0]
        if ok.size == 0:
            continue
        c = ok[rng.integers(ok.size)]
        T[g1], T[g2] = t1[c], t2[c]
        s = np.zeros(64, np.int64)
        for g, tg in zip(groups, T):
            u = np.full(len(g), tg // len(g)) + (np.arange(len(g)) < tg % len(g))
            for _ in range(len(g)):       # texture, same sum
                a, b = rng.choice(len(g), 2, replace=False)
                mv = int(rng.integers(0, 1 + min(u[a] + R, R - u[b])))
                u[a] -= mv
                u[b] += mv
            s[g] = u * np.sign(B[g]).astype(np.int64)
        v = float((B * s).sum())
        if abs(v - target) < tol and np.abs(s).max() <= R:
            return s.reshape(8, 8)
    raise RuntimeError("no sweep block for (%d, %d, %d) at %g" % (cls, i, j, delta))


def sweep_image(seed, HU=32):
    """for every (class, AC position) outside RATIONAL (whose values are multiples of 1/8, so only exact ties come near a
    multiple of q): blocks at the SWEEP distances from the multiple of q at 60 % of the +-R sign pattern of the position,
    and at the SWEEP_T distances around |w| = 1; signs alternate.  Luma blocks fill MCUs four at a time (chroma 0), chroma
    blocks take one MCU each (the other chroma block 0).  -> (r, g, b, W, H)"""
    rng = np.random.default_rng(seed)
    blocks = [[], []]
    for cls, R in ((0, 127), (1, CHROMA_RANGE[1])):
        for n in range(1, 64):
            i, j = divmod(n, 8)
            if (i, j) in RATIONAL:
                continue
            for e, (k, delta) in enumerate([(None, d * (-1) ** t) for t, d in enumerate(SWEEP)] + [(1, d) for d in SWEEP_T]):
                s = sweep_block(rng, cls, i, j, k, delta, R)
                blocks[cls].append(s if (e + n) % 2 else -s)
    nl = -(-len(blocks[0]) // 4)
    cv = Canvas(HU, -(-(nl + len(blocks[1])) // HU))
    for e, s in enumerate(blocks[0]):
        cv.luma(e // 4, e % 4, s)
    for e, s in enumerate(blocks[1]):
        cv.chroma(nl + e, e % 2, s)
    return cv.planes() + (cv.W, cv.H)
