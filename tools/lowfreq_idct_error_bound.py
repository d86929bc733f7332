"""Guard band of the low-frequency class of k_inv_transform2 (jpezy_b200/csrc/dec_transform2.cuh): blocks whose coefficients past
zig-zag position 2 are all zero.  There sample (x, y) is the separable sum

    v = F00 q00 / 8 + 128 + F10 Ly[y] + F01 Lx[x],   Lx[x] = q01 cos((2x+1) pi / 16) / (4 sqrt 2), Ly likewise with q10,

which the kernel evaluates in FP32 (RN) as  p = F00 * M00;  s = p + 128;  base = fma(F10, Ly[y], s);  v = fma(F01, Lx[x], base),
with M00 = q00 / 8 exact and Lx, Ly rounded once from double.  First-order error against the exact sum, with U = 2^-24:

    |v - V| <= U (4 |F00 q00 / 8| + 3 |F10 Ly| + 2 |F01 Lx| + 3 * 128)

(the dequantised DC is rounded in p, s, base and v; F10 Ly in Ly, base and v; F01 Lx in Lx and v; the level shift in s, base and v).
Per unit dequantised coefficient this is E = (4/8, 2 c1, 3 c1) with c1 = cos(pi/16) / (4 sqrt 2); the kernel uses 1.25 E plus
1.25 * 384 U, the margin covering second-order terms and the reference's own FP64 rounding.

The empirical part emulates both sides bit for bit -- the kernel's FP32 operations (the fma exactly in extended precision, then
rounded once) and the reference's FP64 sum in its operation order -- for every sample of coefficient triples with |F| <= 1023
under the Annex K, flat-1 and 255 tables, and checks that the kernel's fast path decides exactly what the reference does
wherever the band lets it decide.  usage: python tools/lowfreq_idct_error_bound.py [--random N]
"""
import argparse
import itertools

import numpy as np

U = 2.0 ** -24
MARGIN = 1.25
C1 = np.cos(np.pi / 16) / (4 * np.sqrt(2.0))
E = np.array([4 / 8, 2 * C1, 3 * C1])          # per unit dequantised coefficient of zig-zag 0, 1 (F01), 2 (F10)
CONST = 3 * 128 * U
# the kernel's constants (dec_transform2.cuh: kLowErrSens0..2 in units of 2^-24, kLowGuard0)
KERNEL_SENS = np.array([0.625, 0.434, 0.651])
KERNEL_CONST = np.float32(2.87e-5)

ANNEX_K_LUMA = [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55]
ANNEX_K_CHROMA = [17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99]
TABLES = {"annexk_luma": ANNEX_K_LUMA, "annexk_chroma": ANNEX_K_CHROMA, "flat1": [1] * 16, "all255": [255] * 16}

COS = np.cos((2 * np.arange(8) + 1) * np.pi / 16)      # cos_ref[8 + k]: the reference's cos((2k+1) * 1 * pi / 16)
INV_SQRT2 = 1.0 / np.sqrt(2.0)


def f32(x):
    return np.asarray(x).astype(np.float32)


def fma32(a, b, c):
    """fma.rn.f32: the exact a * b + c (64-bit mantissa holds it for these operands: checked) rounded once"""
    a, b, c = (np.asarray(t, np.float32).astype(np.longdouble) for t in (a, b, c))
    p = a * b
    s = p + c
    assert np.all((s - p) - c == 0), "extended precision is not exact for these operands"
    return s.astype(np.float32)


def decide(F, q):
    """F: [n, 3] int (zig-zag 0, 1, 2), q: natural table (q[0], q[1], q[8] used).  -> kernel value, guard, reference sample, [n, 8, 8]"""
    q00, q01, q10 = q[0], q[1], q[8]
    s = COS * INV_SQRT2 * 0.25
    lx, ly = f32(q01 * s), f32(q10 * s)
    m00 = np.float32(q00 / 8.0)
    fd, fa, fb = (f32(F[:, k]) for k in range(3))
    # kernel
    p = f32(fd * m00)
    s1 = f32(p + np.float32(128.0))
    base = fma32(fb[:, None], ly[None, :], s1[:, None])                      # [n, y]
    v = fma32(fa[:, None, None], lx[None, None, :], base[:, :, None])        # [n, y, x]
    lg = f32(np.array([q00, q01, q10]) * KERNEL_SENS * U)
    g = fma32(np.abs(fd), lg[0], fma32(np.abs(fa), lg[1], fma32(np.abs(fb), lg[2], KERNEL_CONST)))
    # reference (jpezy_decoder.hpp inverse_dct): natural order (0,0), (0,1), (1,0); ((cu cv) dq) cos cos; int(sum / 4 + 128)
    t0 = (INV_SQRT2 * INV_SQRT2) * (F[:, 0] * q00).astype(np.float64)
    t1 = ((1.0 * INV_SQRT2) * (F[:, 1] * q01).astype(np.float64))[:, None] * COS[None, :]
    t2 = ((INV_SQRT2 * 1.0) * (F[:, 2] * q10).astype(np.float64))[:, None] * COS[None, :]
    tot = (t0[:, None, None] + t1[:, None, :]) + t2[:, :, None]
    ref64 = tot * 0.25 + 128.0
    return v, g, ref64


def check(F, q):
    v, g, ref64 = decide(F, q)
    err = np.abs(v.astype(np.float64) - ref64)
    ratio = float((err / g[:, None, None].astype(np.float64)).max())
    # the fast path: floor(v) when v is at least the band away from every integer and not negative
    dist = np.abs(v - np.round(v))
    fast = (dist >= g[:, None, None]) & (v >= 0)
    wrong = int((np.floor(v[fast]).astype(np.int64) != np.trunc(ref64[fast]).astype(np.int64)).sum())
    return ratio, wrong, int(fast.sum()), v.size


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--random", type=int, default=400000, help="random coefficient triples per table")
    a = ap.parse_args()
    np.set_printoptions(precision=4)
    print("E (2^-24 per unit dequantised coefficient, zig-zag 0, 1, 2):", E, " x margin:", E * MARGIN, " kernel:", KERNEL_SENS)
    print("constant: %.4e, x margin %.4e, kernel %.4e" % (CONST, CONST * MARGIN, KERNEL_CONST))
    assert np.all(KERNEL_SENS >= E * MARGIN) and KERNEL_CONST >= CONST * MARGIN
    rng = np.random.default_rng(5)
    edge = np.array(list(itertools.product([-1023, -1022, -513, -512, -1, 0, 1, 511, 512, 1023], repeat=3)))
    worst = 0.0
    for name, t in TABLES.items():
        q = np.zeros(64, np.int64)
        q[:8], q[8:16] = t[:8], t[8:]
        # every F01 and every F10 against the extreme values of the other two, every DC against them, and random triples
        sweep = np.arange(-1023, 1024)
        ext = np.array([-1023, -1, 0, 1, 1023])
        parts = [edge, rng.integers(-1023, 1024, (a.random, 3))]
        for k in range(3):
            for o1, o2 in itertools.product(ext, ext):
                blk = np.zeros((sweep.size, 3), np.int64)
                blk[:, k] = sweep
                blk[:, (k + 1) % 3], blk[:, (k + 2) % 3] = o1, o2
                parts.append(blk)
        F = np.concatenate(parts)
        tot_ratio, tot_wrong, tot_fast, tot_n = 0.0, 0, 0, 0
        for i in range(0, len(F), 50000):
            r, w, nf, n = check(F[i: i + 50000], q)
            tot_ratio, tot_wrong, tot_fast, tot_n = max(tot_ratio, r), tot_wrong + w, tot_fast + nf, tot_n + n
        worst = max(worst, tot_ratio)
        print("%-14s %8d blocks: max |f32 - ref64| / guard = %.3f ; fast-path samples %d of %d, differing from the reference: %d"
              % (name, len(F), tot_ratio, tot_fast, tot_n, tot_wrong))
        assert tot_wrong == 0 and tot_ratio < 1.0
    print("worst observed error / guard band: %.3f (bound: %.3f)" % (worst, 1 / MARGIN))


if __name__ == "__main__":
    main()
